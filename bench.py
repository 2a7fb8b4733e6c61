#!/usr/bin/env python
"""bench.py — headline benchmark of the dumpvdl2 per-channel DSP hot path on B200.

Metric (BASELINE.json): VDL2 channels demodulated in real time @ 2.1 Msps, reported as whole-job
M channel-samples/s (one channel-sample = one complex input sample processed for one channel);
channels_at_realtime = value / 2.1.

Workload (BASELINE.json config 5, the largest configuration that fits a single B200): 16384 channels per GPU on
64 frequency slots x 256 replicas, fanned out from ONE synthetic 2.1 Msps cu8 stream (Poisson bursts 2/s/slot,
Es/N0 20 dB, SURVEY.md §8d).  One "step" = one pass of the whole path (K0 convert, K1 mix+IIR+decimate, K2a phase,
K2 sync/slice/header, K3 FEC/unstuff/FCS, frames back on the host) over `chunks_per_step` chunks of 262144 IQ pairs
(0.125 s of signal each) for every channel; the default 256 chunks per step make the default K = 6 timed steps a
region of >= 10 s (SURVEY §8d "steady state, >= 10 s").

  --channel-order interleaved (default): channel k sits on slot k mod 64, so the 32 channels of every warp are 32
      different signals (what a deployment looks like); `replica`: the 256 replicas of a slot are adjacent, every warp
      walks 32 copies of one signal and never diverges.  The other order is measured too and printed beside `value`.
  --scaling weak (default): 16384 channels PER GPU; strong: BASELINE config 5 as written, 16384 channels in total,
      channel k on GPU k mod N.  Rank 0 owns the stream; every step's chunks reach the other GPUs through the
      library's multi-GPU ingest helper (vdl2gpu_mg_*: NCCL broadcast or copy-engine peer copies), one step ahead.

  value : chunks resident in HBM before the timed region (N>1: resident on rank 0, the fan-out is timed).
  e2e   : the same metric through the public host-buffer API (Vdl2Channels.process_buf_uchar): host->device copy
          of every chunk and device->host frame records inside the timed region.
  The two legs run A-B-A-B; the first pair gives value / e2e, the second is printed as `repeat`.
  parity: after the timed legs every rank demodulates the first second of the stream once more on ITS shard, hashes
          each channel's (burst, idx, frame octets, FEC corrections, header syndrome weight) list and counters and
          compares them with the oracle (run as a separate checker process on the 64 slot channels); a mismatch
          anywhere makes the benchmark fail.
  --dump-outputs DIR : after the timed legs, what the timed device path delivered for its last step is written to DIR as
          .npy files (see dump_outputs); the inputs depend on the arguments only, so two builds compare output for output.
  --impl reference : the unmodified reference (oracle/_ref/vdl2_ref_fast, one pinned pthread per channel, all host
          threads) on a bounded sample of the same stream; falls back to the oracle port if _ref is absent.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 2100000
OVERSAMPLE = 20
CENTER = 136975000
CHUNK_PAIRS = 262144
CHUNK_BYTES = 2 * CHUNK_PAIRS
N_SLOTS = 64
B_CS = 8.0 + 8.0 / OVERSAMPLE        # algorithmic bytes per channel-sample for K1 (SURVEY.md §8d): 8 B read + 8/os B written
PARITY_CHUNKS = 8                    # the first second of the stream is re-run for the in-bench parity check
METRIC = "VDL2 channel-samples demodulated per second (2.1 Msps channels; real-time channels = value/2.1)"
DUMP_CHANNELS = 512                  # --dump-outputs: fixed, seeded sample of channels whose frames are written
DUMP_BYTES = 64 << 20                # --dump-outputs: cap on all files together
FRAME_FIELDS = ["channel", "burst_seq", "idx", "len", "synd_weight", "datalen_octets", "num_fec_corrections", "fcs_ok",
                "sync_dec_index", "frame_pwr_dbfs", "nf_pwr_dbfs", "ppm_error", "frame_pwr", "mag_nf"]


def make_stream(seconds):
    from dumpvdl2_b200 import synth
    iq, offs, bursts = synth.traffic_stream(FS, seconds, N_SLOTS, 2.0, 20.0, -20.0, 0x56444C33, "u8")
    n_chunks = iq.size // CHUNK_BYTES
    return iq[:n_chunks * CHUNK_BYTES].reshape(n_chunks, CHUNK_BYTES), offs, bursts


def slot_of_channel(n_total, order):
    """global channel index -> frequency slot"""
    k = np.arange(n_total)
    if order == "interleaved":
        return k % N_SLOTS
    reps = -(-n_total // N_SLOTS)
    return np.minimum(k // reps, N_SLOTS - 1)


def channel_freqs(offs, n_total, order="replica"):
    slot = slot_of_channel(n_total, order)
    return (CENTER + np.asarray(offs, dtype=np.int64)[slot]).astype(np.uint32)


# ------------------------------------------------------------------------------------------------------------------
# clocks (NVML in-process: no nvidia-smi child competing for the driver during the timed region)
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, gpu_index, period=0.25):
        self.gpu, self.period, self.rows, self.stop_flag, self.thread, self.h = gpu_index, period, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(gpu_index))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                return i
        return i

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.rows.append((time.time(), sm, mx, reasons, pw))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.nv is None or self.h is None:
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self, t0, t1):
        if self.thread is None:
            return None
        self.stop_flag = True
        self.thread.join(timeout=2)
        rows = [r for r in self.rows if t0 <= r[0] <= t1] or self.rows
        if not rows:
            return None
        sm = sorted(r[1] for r in rows)
        bits = 0
        for r in rows:
            bits |= int(r[3])
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        return dict(sm_mhz=float(sm[len(sm) // 2]), sm_min_mhz=float(sm[0]), sm_max_mhz=float(rows[0][2]),
                    reasons=[n for b, n in names.items() if bits & b], samples=len(rows), power_w_max=max(r[4] for r in rows),
                    source="NVML in-process, 4 Hz, during the first timed leg")


# ------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline
# ------------------------------------------------------------------------------------------------------------------
def _ref_passes(chunks, offs, passes, loops):
    """oracle/_ref/vdl2_ref_fast (the unmodified reference) on a bounded sample: returns (n_ch, cores, [M ch-samples/s per pass])"""
    from oracle import pyoracle as po
    cores = os.cpu_count() or 1
    n_ch = max(1, min(cores - 1 if cores > 1 else 1, 256))
    freqs = channel_freqs(offs, n_ch, "interleaved")
    with tempfile.NamedTemporaryFile(suffix=".cu8", delete=False) as tf:
        tf.write(chunks.tobytes())
        path = tf.name
    vals = []
    try:
        for _ in range(passes):
            _, st = po.run_ref(path, po.FMT_U8, OVERSAMPLE, CENTER, freqs, flavour="fast", chunk=CHUNK_BYTES, quiet=True, loop=loops, pin=True)
            vals.append(st["ch_msamples_per_s"])
    finally:
        os.unlink(path)
    return n_ch, cores, vals


def cpu_baseline_leg(passes=3):
    """Bounded (~10-30 s) timing of the reference CPU path on this host, reported beside the GPU numbers: median of
    `passes` runs, one pinned thread per channel."""
    from oracle import pyoracle as po
    chunks, offs, _ = make_stream(1.0)
    cores = os.cpu_count() or 1
    if po.ref_binary("fast"):
        loops = 2
        n_ch, cores, vals = _ref_passes(chunks, offs, passes, loops)
        v = float(np.median(vals))
        return dict(value=v, unit="Msamples/s", cores=n_ch + 1, kind="reference", host_cpus=cores, passes=[round(x, 1) for x in vals],
                    sample=f"{n_ch} channels (one pinned pthread each + 1 producer) x {loops} x {chunks.size / 2 / FS:.2f} s of the bench stream, "
                           f"median of {passes} passes, unmodified reference built -O2 -ffast-math", channels_at_realtime=v / 2.1)
    n_ch = 4
    o = po.Oracle(FS, OVERSAMPLE, po.FMT_U8, CENTER, channel_freqs(offs, n_ch, "interleaved"))
    t0 = time.time(); o.process_chunked(chunks.reshape(-1), CHUNK_BYTES); dt = time.time() - t0
    v = n_ch * chunks.size / 2 / dt / 1e6
    return dict(value=v, unit="Msamples/s", cores=1, kind="port", host_cpus=cores,
                sample=f"{n_ch} channels x {chunks.size / 2 / FS:.2f} s, single-thread oracle port", channels_at_realtime=v / 2.1)


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path on this host's cores; a step = one pass of
    all channel threads over the bounded sample."""
    if rank != 0:
        return
    from oracle import pyoracle as po
    chunks, offs, _ = make_stream(1.0)
    cores = os.cpu_count() or 1
    per = []
    if po.ref_binary("fast"):
        kind = "reference"
        loops = 4
        n_ch, cores, vals = _ref_passes(chunks, offs, args.warmup + args.steps, loops)
        per = vals[args.warmup:]
        threads = n_ch + 1
        how = "one pinned pthread per channel + producer"
    else:
        kind, n_ch, threads, how, loops = "port", 4, 1, "single-thread oracle port", 1
        for step in range(args.warmup + args.steps):
            o = po.Oracle(FS, OVERSAMPLE, po.FMT_U8, CENTER, channel_freqs(offs, n_ch, "interleaved"))
            t0 = time.time(); o.process_chunked(chunks.reshape(-1), CHUNK_BYTES); dt = time.time() - t0
            if step >= args.warmup:
                per.append(n_ch * chunks.size / 2 / dt / 1e6)
    value = float(np.median(per))
    sample_pairs = loops * chunks.size // 2
    sample = f"{n_ch} channels x {sample_pairs / FS:.2f} s of the bench stream per step ({how}); value = median over the timed steps"
    line = dict(impl="reference", metric=METRIC, value=value, unit="Msamples/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=n_ch * sample_pairs / value / 1e3, higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f32",
                data="synthetic",
                config=dict(workload=f"reference CPU path on a bounded sample: {sample}", fs=FS, oversample=OVERSAMPLE,
                            channels=n_ch, sample_fmt="cu8", l2="n/a (CPU)"),
                channels_at_realtime=value / 2.1, per_step=[round(x, 1) for x in per],
                cpu_baseline=dict(value=value, unit="Msamples/s", cores=threads, kind=kind, sample=sample, host_cpus=cores),
                e2e=dict(value=value, unit="Msamples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, frames, counters, first_dec, suffix=""):
    """--dump-outputs: the frames the timed device path delivered for its last step and the per-channel counters after it.

    frames_meta.npy      float64 [n, len(FRAME_FIELDS)]: one row per frame, columns FRAME_FIELDS (every value exact)
    frames_data.npy      float32 [sum of len]: the frames' octets back to back, in row order
    frames_channels.npy  float64: the sampled channels, sorted
    channel_counters.npy float64 [channels, 9]: api.COUNTER_NAMES per channel, cumulative over the whole leg
    Frames are those synced in the last step (sync_dec_index >= first_dec: which poll of the pipeline hands over a frame
    near a step boundary depends on timing, where its burst was synced does not) on a fixed, seeded sample of
    DUMP_CHANNELS channels, sorted by (channel, burst, idx) and cut where the files would exceed DUMP_BYTES."""
    n_ch = counters.shape[0]
    sample = np.sort(np.random.default_rng(0x56444C33).choice(n_ch, min(DUMP_CHANNELS, n_ch), replace=False))
    keep = set(int(c) for c in sample)
    budget = DUMP_BYTES - counters.size * 8 - sample.size * 8
    rows, data = [], []
    for f in sorted((f for f in frames if f.channel in keep and f.sync_dec_index >= first_dec), key=lambda f: f.key()):
        budget -= len(FRAME_FIELDS) * 8 + len(f.data) * 4
        if budget < 0:
            break
        rows.append([float(getattr(f, k)) if k != "len" else float(len(f.data)) for k in FRAME_FIELDS])
        data.append(np.frombuffer(f.data, np.uint8))
    os.makedirs(out_dir, exist_ok=True)
    meta = np.array(rows, np.float64).reshape(-1, len(FRAME_FIELDS))
    np.save(os.path.join(out_dir, f"frames_meta{suffix}.npy"), meta)
    np.save(os.path.join(out_dir, f"frames_data{suffix}.npy"), (np.concatenate(data) if data else np.zeros(0, np.uint8)).astype(np.float32))
    np.save(os.path.join(out_dir, f"frames_channels{suffix}.npy"), sample.astype(np.float64))
    np.save(os.path.join(out_dir, f"channel_counters{suffix}.npy"), counters.astype(np.float64))
    print(f"--dump-outputs: {meta.shape[0]} frames of {sample.size} channels, counters of {n_ch} channels -> {out_dir}", file=sys.stderr)


# ------------------------------------------------------------------------------------------------------------------
# parity checker (the oracle runs in its own process: nothing under oracle/ is loaded into the measured process)
# ------------------------------------------------------------------------------------------------------------------
def digest_frames(frames, counters_row):
    h = hashlib.sha256()
    for f in sorted(frames, key=lambda f: (f.burst_seq, f.idx)):
        h.update(f"{f.burst_seq},{f.idx},{f.num_fec_corrections},{f.synd_weight},{f.data.hex()};".encode())
    h.update(",".join(str(int(x)) for x in counters_row).encode())
    return h.hexdigest()


def oracle_digest_main(path_in, path_out):
    """hidden mode (--oracle-digest): oracle over the 64 slot channels of the parity sample -> per-slot digests"""
    from oracle import pyoracle as po
    with open(path_in, "rb") as f:
        meta = json.loads(f.readline().decode())
        iq = np.frombuffer(f.read(), np.uint8)
    o = po.Oracle(FS, OVERSAMPLE, po.FMT_U8, CENTER, np.asarray(meta["freqs"], dtype=np.uint32))
    o.process_chunked(iq, CHUNK_BYTES)
    by = {}
    for f in o.frames():
        by.setdefault(f.channel, []).append(f)
    cnt = o.counters()
    out = dict(digests=[digest_frames(by.get(s, []), cnt[s]) for s in range(len(meta["freqs"]))],
               frames=sum(len(v) for v in by.values()))
    with open(path_out, "w") as f:
        json.dump(out, f)


def oracle_slot_digests(chunks, offs):
    with tempfile.TemporaryDirectory() as td:
        pin, pout = os.path.join(td, "in.bin"), os.path.join(td, "out.json")
        with open(pin, "wb") as f:
            f.write((json.dumps(dict(freqs=[int(CENTER + int(o)) for o in offs])) + "\n").encode())
            f.write(chunks[:PARITY_CHUNKS].tobytes())
        subprocess.run([sys.executable, os.path.abspath(__file__), "--oracle-digest", pin, pout], check=True)
        with open(pout) as f:
            return json.load(f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--channels", type=int, default=16384, help="channels per GPU (weak scaling) / in total (strong scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--channel-order", default="interleaved", choices=["interleaved", "replica"])
    ap.add_argument("--chunks-per-step", type=int, default=256)
    ap.add_argument("--stream-seconds", type=float, default=4.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-repeat", action="store_true", help="skip the second value/e2e pair and the other channel order")
    ap.add_argument("--k1-scalar", action="store_true")
    ap.add_argument("--fanout", default="nccl", choices=["auto", "nccl", "ce"], help="multi-GPU ingest: NCCL broadcast (default) or copy-engine peer copies")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step to DIR/*.npy")
    ap.add_argument("--oracle-digest", nargs=2, metavar=("IN", "OUT"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.oracle_digest:
        oracle_digest_main(*args.oracle_digest)
        return
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    # keep stdout clean for the single JSON line: libraries (NCCL prints its version banner there) write to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    import dumpvdl2_b200 as vd
    from dumpvdl2_b200 import shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the demodulator path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    W, K, CPS = max(args.warmup, 3), args.steps, args.chunks_per_step
    n_total = args.channels * world if args.scaling == "weak" else args.channels
    chunks, offs, bursts = make_stream(args.stream_seconds)       # same seed on every rank
    n_chunks = chunks.shape[0]
    flags = vd.FLAG_K1_SCALAR if args.k1_scalar else 0
    stream = torch.cuda.current_stream()

    def make_ctx(order, extra_flags=0):
        all_freqs = channel_freqs(offs, n_total, order)
        mine = shard.my_channels(all_freqs, rank, world)          # channel k -> GPU k mod N
        return vd.Vdl2Channels(FS, OVERSAMPLE, vd.FMT_U8, CENTER, mine, max_chunk_bytes=CHUNK_BYTES, device=local_rank,
                               flags=flags | extra_flags), mine

    g, my_freqs = make_ctx(args.channel_order)
    n_mine = len(my_freqs)

    # chunks resident in HBM on the ingest rank (rank 0) and in pinned host memory
    d_chunks = torch.from_numpy(chunks).cuda()          # every rank keeps a copy for the local kernel timing; rank 0's is the fan-out source
    h_chunks = torch.from_numpy(chunks).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: the library's multi-GPU ingest helper owns the double-buffered receive area and the fan-out
    mg = shard.MultiGpuIngest(g, rank, world, CPS * CHUNK_BYTES, mode=args.fanout) if world > 1 else None
    state = dict(chunk=0)

    def next_indices():
        idx = [(state["chunk"] + k) % n_chunks for k in range(CPS)]
        state["chunk"] += CPS
        return idx

    host_t = dict(submit_s=0.0, submits=0)

    def gather_rows(src, idx):
        """[(ptr, nbytes)] of the contiguous runs of rows idx in src (device- or pinned-host-resident tensor)"""
        runs, k = [], 0
        while k < len(idx):
            j = k
            while j + 1 < len(idx) and idx[j + 1] == idx[j] + 1:
                j += 1
            runs.append((src[idx[k]].data_ptr(), (j + 1 - k) * CHUNK_BYTES))
            k = j + 1
        return runs

    def step_multi(src_rows, src_is_host, harvest=True):
        """stage step s+1 (rank 0 gathers the chunks into the free half of the receive area, all ranks take part in the
        fan-out) BEFORE the chunks of step s are submitted: the transfer overlaps the kernels.  A staged step is always
        consumed, also across the legs of the benchmark (its bytes are the same whichever memory they came from)."""
        if state.get("staged") is None:
            state["staged"] = mg.stage(gather_rows(src_rows, next_indices()) if rank == 0 else None, src_is_host)
        buf = state["staged"]
        state["staged"] = mg.stage(gather_rows(src_rows, next_indices()) if rank == 0 else None, src_is_host)
        t0 = time.perf_counter()
        mg.submit_staged(buf, CPS, CHUNK_BYTES)
        host_t["submit_s"] += time.perf_counter() - t0; host_t["submits"] += CPS
        return g.poll_count() if harvest else 0

    def step_device(harvest=True):
        """one step, chunks already in HBM (N>1: fanned out from rank 0, one step ahead)"""
        if world > 1:
            return step_multi(d_chunks if rank == 0 else None, False, harvest)
        t0 = time.perf_counter()
        for i in next_indices():
            g.submit_device(d_chunks[i].data_ptr(), CHUNK_BYTES, stream.cuda_stream)
        host_t["submit_s"] += time.perf_counter() - t0; host_t["submits"] += CPS
        return g.poll_count() if harvest else 0

    def step_host(harvest=True):
        """one step through the public host-buffer entry point (process_buf_uchar); with N > 1 the ingest rank copies
        the step's chunks host->device and fans them out, the other ranks receive"""
        if world > 1:
            return step_multi(h_chunks, True, harvest)
        hn = h_chunks.numpy()
        t0 = time.perf_counter()
        for i in next_indices():
            g.process_buf_uchar(hn[i])
        host_t["submit_s"] += time.perf_counter() - t0; host_t["submits"] += CPS
        return g.poll_count() if harvest else 0

    def timed(step_fn, steps, sample_clocks=False, capture=False):
        """capture: the last step's frames are not harvested inside the timed region; the region ends when the device has
        drained, and they are collected after it (r["captured"])"""
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        barrier()
        s0 = g.stats()
        host_t["submit_s"], host_t["submits"] = 0.0, 0
        if sampler:
            sampler.start()
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 2)]
        t0 = time.time()
        ev[0].record(stream)
        frames = 0
        for k in range(steps):
            frames += step_fn(not (capture and k == steps - 1))     # submits + non-blocking harvest: the pipeline stays full across steps
            g.stream_wait(stream.cuda_stream)
            ev[k + 1].record(stream)     # completes when every kernel of steps 0..k has run
        if not capture:
            frames += g.flush_count()    # everything submitted is processed and its frames are on the host
        g.stream_wait(stream.cuda_stream)
        ev[steps + 1].record(stream)
        barrier()
        t1 = time.time()
        captured = None
        if capture:
            captured = dict(frames=g.flush(), counters=g.channel_counters(),
                            first_dec=(s0["iq_samples"] + (steps - 1) * CPS * CHUNK_PAIRS) // OVERSAMPLE + 1)
            frames += len(captured["frames"])
        ms = ev[0].elapsed_time(ev[steps + 1])
        per = [ev[k].elapsed_time(ev[k + 1]) for k in range(steps)]
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        clocks = sampler.stop(t0, t1) if sampler else None
        s1 = g.stats()
        return dict(ms=ms, per_step=per, frames=frames, d={k: s1[k] - s0[k] for k in s1}, clocks=clocks, wall_ms=(t1 - t0) * 1e3,
                    host_us_per_submit=host_t["submit_s"] / max(host_t["submits"], 1) * 1e6, captured=captured)

    def leg(kind, steps, warm, sample_clocks=False, capture=False):
        fn = step_device if kind == "device" else step_host
        for _ in range(warm):
            fn()
        g.flush_count()
        r = timed(fn, steps, sample_clocks, capture)
        g.flush_count()
        return r

    cs_per_step = float(n_total) * CPS * CHUNK_PAIRS

    def rate(r, steps):
        return cs_per_step * steps / (r["ms"] * 1e-3) / 1e6

    # ---- A-B-A-B ----
    A1 = leg("device", K, W, sample_clocks=True, capture=bool(args.dump_outputs))
    if args.dump_outputs:
        cap = A1.pop("captured")
        dump_outputs(args.dump_outputs, cap["frames"], cap["counters"], cap["first_dec"], f"_rank{rank}" if world > 1 else "")
        del cap
    B1 = leg("host", K, 1)
    A2 = B2 = None
    if not args.no_repeat:
        A2 = leg("device", K, 1)
        B2 = leg("host", K, 1)

    # ---- the other channel order, same code path, a shorter region ----
    other = None
    if not args.no_repeat:
        other_order = "replica" if args.channel_order == "interleaved" else "interleaved"
        g_main, mg_main, staged_main = g, mg, state.get("staged")
        state["staged"] = None
        g, _ = make_ctx(other_order)
        if world > 1:
            mg = shard.MultiGpuIngest(g, rank, world, CPS * CHUNK_BYTES, mode=args.fanout)
        ko = max(2, K // 2)
        r = leg("device", ko, 1)
        other = dict(order=other_order, value=rate(r, ko), ms_per_step=r["ms"] / ko)
        if world > 1:
            mg.close()
        g.close()
        g, mg = g_main, mg_main
        state["staged"] = staged_main

    # ---- per-kernel durations for the roofline: the production pipeline runs K0/K1 of chunk c+1 beside K2/K3 of chunk c
    # on two streams, which stretches every kernel's wall time; the kernel's OWN launch duration is therefore measured here,
    # live, with CUDA events on the library's streams, same workload, same process, with that overlap switched off
    # (VDL2GPU_FLAG_NO_OVERLAP) - the condition the committed ncu launch list is taken under as well.
    kms, ms_serial, n_serial = None, None, 0
    if True:                             # at any N: every rank times its own kernels on locally resident chunks (no fan-out involved)
        g_main = g
        g, _ = make_ctx(args.channel_order, vd.FLAG_NO_OVERLAP)
        for _ in range(8):
            g.submit_device(d_chunks[_ % n_chunks].data_ptr(), CHUNK_BYTES, stream.cuda_stream)
        g.flush_count()
        g.enable_timing(True)
        k0 = g.kernel_ms()
        n_serial = 48
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(n_serial):
            g.submit_device(d_chunks[i % n_chunks].data_ptr(), CHUNK_BYTES, stream.cuda_stream)
            g.poll_count()
        g.flush_count()
        g.stream_wait(stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_serial = e0.elapsed_time(e1) / n_serial
        k1 = g.kernel_ms()
        g.close()
        g = g_main
        kms = {k: ((k1[k][0] - k0[k][0]) / max(k1[k][1] - k0[k][1], 1)) for k in k1}

    # ---- parity: every rank re-runs the first second on its shard and compares with the oracle's slot channels ----
    parity = None
    if not args.no_parity:
        ref = None
        if rank == 0:
            ref = oracle_slot_digests(chunks, offs)
        if world > 1:
            box = [ref]
            dist.broadcast_object_list(box, src=0)
            ref = box[0]
        gp, mine = make_ctx(args.channel_order)
        for i in range(PARITY_CHUNKS):
            gp.process_buf_uchar(chunks[i])
        by = {}
        for f in gp.flush():
            by.setdefault(f.channel, []).append(f)
        cnt = gp.channel_counters()
        gp.close()
        slot = slot_of_channel(n_total, args.channel_order)[rank::world]
        mism, frames_checked = 0, 0
        for j in range(len(mine)):
            fr = by.get(j, [])
            frames_checked += len(fr)
            if digest_frames(fr, cnt[j]) != ref["digests"][int(slot[j])]:
                mism += 1
        tot = torch.tensor([mism, len(mine), frames_checked, 1], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(tot)
        parity = dict(ranks_checked=int(tot[3]), channels_checked=int(tot[1]), frames_checked=int(tot[2]), mismatches=int(tot[0]),
                      oracle_frames_per_slot_set=ref["frames"], seconds=PARITY_CHUNKS * CHUNK_PAIRS / FS,
                      what="per-channel (burst, idx, frame octets, FEC corrections, syndrome weight) lists + 9 counters vs the oracle port")

    value = rate(A1, K)
    e2e_value = rate(B1, K)

    if rank == 0:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peak = float(json.load(f)["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json, burst copy)"
        except Exception:
            pass
        prof = {}
        try:
            with open(os.path.join(ROOT, "profiles", "kernel_counters.json")) as f:
                prof = json.load(f)
        except Exception:
            pass
        roofline = None
        if kms:
            k1_ms = kms["K1"]
            achieved = n_mine * CHUNK_PAIRS * B_CS / (k1_ms * 1e-3) / 1e9 if k1_ms > 0 else None
            tot_k = sum(kms.values()) or 1.0
            n_dec = CHUNK_PAIRS // OVERSAMPLE
            sm_clock = 1.965e9
            smsp = 148 * 4
            traffic = None
            tj = prof.get("K1", {})
            if tj.get("channels") == n_mine and tj.get("chunk_pairs") == CHUNK_PAIRS:
                traffic = tj.get("dram_bytes_per_launch")
            stages = {}
            for name in ("K1", "K2a", "K2", "K3"):
                pj = prof.get(name, {})
                ent = dict(ms_per_launch=kms[name], share_of_step=kms[name] / tot_k)
                wi = pj.get("warp_instructions_per_launch")
                if wi and pj.get("channels") == n_mine and kms[name] > 0:
                    # issue-slot model: warp-instructions issued / (SM sub-partitions x clock x duration)
                    ent["issue_slots"] = dict(warp_instructions=wi, frac=wi / (smsp * sm_clock * kms[name] * 1e-3),
                                              per_decimated_sample_per_warp=wi / (n_dec * -(-n_mine // 32)))
                if pj.get("dram_bytes_per_launch") and pj.get("channels") == n_mine:
                    ent["dram_gbs"] = pj["dram_bytes_per_launch"] / (kms[name] * 1e-3) / 1e9
                    ent["dram_frac_of_peak"] = ent["dram_gbs"] / peak
                stages[name] = ent
            fp32 = n_mine * CHUNK_PAIRS * 24.0 / (k1_ms * 1e-3)
            roofline = dict(bound="hbm", kernel="k1_mix_iir_decimate", achieved=achieved, peak=peak, unit="GB/s",
                            frac=(achieved / peak) if achieved else None, traffic=traffic, peak_source=peak_src,
                            bytes_per_channel_sample=B_CS, ms_per_launch=k1_ms,
                            note="SURVEY §8d effective-bandwidth model (each channel streams the float IQ buffer: 8.4 B per channel-sample). "
                                 "It is NOT HBM utilisation: the shared stream is staged once per warp in shared memory (TMA), real DRAM traffic "
                                 "is `traffic`; the bound that binds K1 is `binding` (FP32 issue of one warp per SM sub-partition)",
                            binding=dict(bound="fp32-issue", achieved=fp32 / 1e12, peak=148 * 128 * sm_clock / 1e12, unit="T lane-ops/s",
                                         frac=fp32 / (148 * 128 * sm_clock),
                                         note="24 individually rounded FP32 operations per channel-sample (11 packed FMUL2/FFMA2 + 2 scalar; contraction is "
                                              "not allowed by the bit-exactness contract) against 148 SMs x 128 FP32 lanes x 1.965 GHz.  One warp per "
                                              "sub-partition with 27-28 of its 32 lanes holding a channel (16384 channels dealt over 592 warps) caps this at "
                                              "0.86; a packed operation blocks the issuing warp for 2.25 cycles, so the instruction mix costs ~33 cycles per "
                                              "sample per warp (36.7 measured) against 24 at the pipe's peak"),
                            stages=stages,
                            measured="CUDA events on the library's streams, kernels serialised (VDL2GPU_FLAG_NO_OVERLAP, kernel-by-kernel "
                                     "launches), same workload and process; value/e2e run the two-stage overlap with CUDA graph replay",
                            serial_ms_per_chunk=ms_serial, sum_kernel_ms_per_chunk=tot_k)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu = cpu_baseline_leg()
            except Exception as ex:          # the baseline is a report, never a dependency of the GPU path
                cpu = dict(error=str(ex))

        def stat(per):
            s = sorted(per)
            return dict(min=s[0], median=s[len(s) // 2], max=s[-1])
        line = dict(
            metric=METRIC, value=value, unit="Msamples/s", n_gpus=world, steps=K, warmup=W, ms_per_step=A1["ms"] / K,
            higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f32", data="synthetic",
            config=dict(workload=f"{n_mine} channels/GPU ({n_total} total) on 64 slots from one synthetic 2.1 Msps cu8 stream "
                                 f"(BASELINE config 5; Poisson bursts 2/s/slot, Es/N0 20 dB); step = {CPS} chunks x {CHUNK_PAIRS} IQ pairs "
                                 f"= {CPS * CHUNK_PAIRS / FS:.1f} s of signal per channel",
                        fs=FS, oversample=OVERSAMPLE, channels_per_gpu=n_mine, channels_total=n_total, sample_fmt="cu8",
                        chunk_pairs=CHUNK_PAIRS, chunks_per_step=CPS, channel_order=args.channel_order,
                        parallelism=(f"channel-shard x{world} (k mod N), {mg.mode_name} fan-out of the IQ chunks" if world > 1 else "single GPU"),
                        l2=f"inputs larger than L2: the per-chunk working set (decimated buffer {n_mine * (CHUNK_PAIRS // OVERSAMPLE) * 8 / 1e6:.0f} MB "
                           f"written by K1, read by K2a/K2, + phase plane) exceeds the 126 MB L2 and is rewritten every chunk",
                        k1_impl="scalar" if args.k1_scalar else "pipelined f32x2",
                        pipeline="two streams in lock step: K2a of chunk c alone (phase pass, full occupancy), then K0/K1 of chunk c+1 beside K2/K3 of chunk c, one block per SM each; three CUDA graph replays per chunk"),
            channels_at_realtime=value / 2.1,
            frames_per_step=A1["frames"] / K,
            step_ms=stat(A1["per_step"]), host_us_per_submit=A1["host_us_per_submit"],
            timed_region_s=A1["ms"] / 1e3,
            e2e=dict(value=e2e_value, unit="Msamples/s", h2d_bytes_per_step=CPS * CHUNK_BYTES,
                     d2h_bytes_per_step=B1["d"]["out_bytes"] / K, ms_per_step=B1["ms"] / K, channels_at_realtime=e2e_value / 2.1,
                     frames_per_step=B1["frames"] / K, step_ms=stat(B1["per_step"]), host_us_per_submit=B1["host_us_per_submit"],
                     api="Vdl2Channels.process_buf_uchar (vdl2gpu_submit) + poll/flush"),
            gpu_launches=int(A1["d"]["kernel_launches"]), graph_launches=int(A1["d"]["graph_launches"]),
            clocks=A1["clocks"],
            counts=dict(pool_overflows=int(A1["d"]["pool_overflows"] + B1["d"]["pool_overflows"]), out_overflows=int(A1["d"]["out_overflows"] + B1["d"]["out_overflows"]),
                        bursts_per_step=A1["d"]["bursts"] / K, fcs_good_per_step=A1["d"]["fcs_good"] / K, fcs_bad_per_step=A1["d"]["fcs_bad"] / K),
            wall_ms_per_step=A1["wall_ms"] / K,
        )
        if A2 is not None:
            line["repeat"] = dict(value=rate(A2, K), e2e=rate(B2, K), value_rel_diff=rate(A2, K) / value - 1.0,
                                  e2e_rel_diff=rate(B2, K) / e2e_value - 1.0, order="A-B-A-B, this is the second pair")
        if other is not None:
            line["value_" + other["order"].replace("replica", "replica_adjacent")] = other["value"]
            line["other_channel_order"] = other
        if roofline is not None:
            line["roofline"] = roofline
        if parity is not None:
            line["parity"] = parity
        if cpu is not None:
            line["cpu_baseline"] = cpu
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    barrier()
    if mg is not None:
        mg.close()
    g.close()
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and parity["mismatches"] != 0:
        sys.exit(3)


if __name__ == "__main__":
    main()
