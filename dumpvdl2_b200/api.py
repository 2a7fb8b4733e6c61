"""Python face of libvdl2gpu.so (ctypes over the C-ABI in include/vdl2gpu.h).

The names mirror the reference's interface for this path: a `Vdl2Channels` object is the set of
vdl2_channel_t's created by vdl2_channel_init (src/demod.c:379-392); `process_buf_uchar` /
`process_buf_short` (src/demod.c:339-365) feed it; frames come back with the metadata of
decode_frame / vdl2_msg_metadata (src/decode.c:173-194, src/output-common.h:31-43) instead of through
avlc_decoder_queue_push.  There is no CPU path: constructing the object without the built extension or
without a B200 raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvdl2gpu.so")
FMT_U8, FMT_S16 = 0, 1
FLAG_TRACE, FLAG_KEEP_DEC, FLAG_K1_SCALAR, FLAG_NO_OVERLAP, FLAG_NO_GRAPH = 1, 2, 4, 8, 16
NUM_COUNTERS = 9
COUNTER_NAMES = ["sync_good", "hdr_crc_good", "bursts", "burst_err", "blocks_processed",
                 "blocks_fec_ok", "msg_good", "fcs_good", "fcs_bad"]


class Vdl2GpuError(RuntimeError):
    pass


class _Timeval(C.Structure):
    _fields_ = [("tv_sec", C.c_long), ("tv_usec", C.c_long)]


class _Config(C.Structure):
    _fields_ = [("sample_rate", C.c_uint32), ("oversample", C.c_uint32), ("sample_fmt", C.c_uint32),
                ("centerfreq", C.c_uint32), ("n_channels", C.c_uint32), ("freqs", C.POINTER(C.c_uint32)),
                ("max_ppm", C.c_float), ("max_chunk_bytes", C.c_uint32), ("device", C.c_int32),
                ("flags", C.c_uint32), ("n_inflight", C.c_uint32), ("n_streams", C.c_uint32), ("reserved", C.c_uint32 * 4)]


class _StreamLayout(C.Structure):
    _fields_ = [("n_streams", C.c_uint32), ("channels_per_stream", C.POINTER(C.c_uint32)), ("centerfreqs", C.POINTER(C.c_uint32))]


class _Frame(C.Structure):
    _fields_ = [("channel", C.c_uint32), ("freq", C.c_uint32), ("burst_seq", C.c_uint32), ("idx", C.c_int32),
                ("data", C.POINTER(C.c_uint8)), ("len", C.c_uint32), ("synd_weight", C.c_uint32),
                ("datalen_octets", C.c_uint32), ("num_fec_corrections", C.c_int32),
                ("frame_pwr_dbfs", C.c_float), ("nf_pwr_dbfs", C.c_float), ("ppm_error", C.c_float),
                ("frame_pwr", C.c_float), ("mag_nf", C.c_float), ("sync_dec_index", C.c_uint64),
                ("burst_timestamp", _Timeval), ("fcs_residue", C.c_uint16), ("fcs_ok", C.c_uint16)]


class _Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in
                ("chunks_submitted", "chunks_completed", "iq_samples", "dec_samples", "demod_sync_good",
                 "decoder_crc_good", "bursts", "burst_errors", "blocks_processed", "blocks_fec_ok", "msg_good",
                 "fcs_good", "fcs_bad", "pool_overflows", "out_overflows", "kernel_launches", "out_bytes", "graph_launches")] + [("reserved", C.c_uint64 * 2)]


class _Event(C.Structure):
    _fields_ = [("channel", C.c_uint32), ("kind", C.c_uint32), ("dec_index", C.c_uint64),
                ("i", C.c_int32 * 8), ("f", C.c_float * 8)]


_FRAME_CB = C.CFUNCTYPE(None, C.POINTER(_Frame), C.c_void_p)
_LIB = None


def load_library():
    """Load libvdl2gpu.so; raises if it has not been built (python -m dumpvdl2_b200.build)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise Vdl2GpuError(f"{LIB_PATH} is missing: build it with `python -m dumpvdl2_b200.build` "
                           "(nvcc, sm_100a). There is no CPU fallback for the demodulator path.")
    L = C.CDLL(LIB_PATH)
    L.vdl2gpu_create.argtypes = [C.POINTER(_Config), C.POINTER(C.c_void_p)]
    L.vdl2gpu_create_streams.argtypes = [C.POINTER(_Config), C.POINTER(_StreamLayout), C.POINTER(C.c_void_p)]
    L.vdl2gpu_destroy.argtypes = [C.c_void_p]
    L.vdl2gpu_submit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.vdl2gpu_submit_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.vdl2gpu_submit_planar_s16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
    L.vdl2gpu_serialize_raw_frame.argtypes = [C.POINTER(_Frame), C.c_char_p, C.c_void_p, C.c_size_t]
    L.vdl2gpu_wait_input_consumed.argtypes = [C.c_void_p, C.c_void_p]
    L.vdl2gpu_stream_wait.argtypes = [C.c_void_p, C.c_void_p]
    L.vdl2gpu_poll.argtypes = [C.c_void_p, _FRAME_CB, C.c_void_p]
    L.vdl2gpu_flush.argtypes = [C.c_void_p, _FRAME_CB, C.c_void_p]
    L.vdl2gpu_get_stats.argtypes = [C.c_void_p, C.POINTER(_Stats)]
    L.vdl2gpu_get_channel_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.vdl2gpu_get_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 8
    L.vdl2gpu_read_dec.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32)]
    L.vdl2gpu_read_events.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.vdl2gpu_enable_timing.argtypes = [C.c_void_p, C.c_int]
    L.vdl2gpu_get_kernel_ms.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.vdl2gpu_get_timeline.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.vdl2gpu_debug_block_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.vdl2gpu_strerror.restype = C.c_char_p
    L.vdl2gpu_strerror.argtypes = [C.c_int]
    L.vdl2gpu_last_error.restype = C.c_char_p
    L.vdl2gpu_launch_convert.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.vdl2gpu_launch_fcs_crc16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    L.vdl2gpu_launch_rs_verify.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    L.vdl2gpu_launch_phase_mag.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.vdl2gpu_chunks_in_flight.argtypes = [C.c_void_p]
    L.vdl2gpu_stage_device_bytes.restype = C.c_size_t
    L.vdl2gpu_stage_device_bytes.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32]
    L.vdl2gpu_stage_row_stride.restype = C.c_uint32
    L.vdl2gpu_stage_row_stride.argtypes = [C.c_uint32]
    L.vdl2gpu_stage_create.argtypes = [C.POINTER(_Config), C.c_uint32, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.vdl2gpu_stage_destroy.argtypes = [C.c_void_p]
    L.vdl2gpu_stage_levels.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.vdl2gpu_launch_mix_iir_decimate.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p]
    L.vdl2gpu_launch_sync_slice.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.vdl2gpu_launch_burst_fec.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.vdl2gpu_parse_records.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, _FRAME_CB, C.c_void_p]
    L.vdl2gpu_stage_read_events.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    _LIB = L
    return L


def _check(L, rc, what):
    if rc < 0:
        raise Vdl2GpuError(f"{what}: {L.vdl2gpu_strerror(rc).decode()} ({L.vdl2gpu_last_error().decode()})")
    return rc


class Frame:
    """One AVLC frame + vdl2_msg_metadata fields (src/output-common.h:31-43)."""
    __slots__ = ("channel", "freq", "burst_seq", "idx", "data", "synd_weight", "datalen_octets",
                 "num_fec_corrections", "frame_pwr_dbfs", "nf_pwr_dbfs", "ppm_error", "frame_pwr", "mag_nf",
                 "sync_dec_index", "burst_timestamp", "fcs_ok")

    def key(self):
        return (self.channel, self.burst_seq, self.idx)

    def __repr__(self):
        return (f"Frame(ch={self.channel} burst={self.burst_seq} idx={self.idx} len={len(self.data)} "
                f"fcs_ok={self.fcs_ok} fec={self.num_fec_corrections} synd={self.synd_weight})")


def serialize_raw_frame(frame, station_id=None, timestamp=(0, 0)):
    """Frame -> one record of the reference's raw-frame archive format (see vdl2gpu_serialize_raw_frame)."""
    L = load_library()
    f = _Frame()
    buf = (C.c_uint8 * max(len(frame.data), 1)).from_buffer_copy(frame.data or b"\0")
    f.channel, f.freq, f.burst_seq, f.idx = frame.channel, frame.freq, frame.burst_seq, frame.idx
    f.data, f.len = C.cast(buf, C.POINTER(C.c_uint8)), len(frame.data)
    f.synd_weight, f.datalen_octets, f.num_fec_corrections = frame.synd_weight, frame.datalen_octets, frame.num_fec_corrections
    f.frame_pwr_dbfs, f.nf_pwr_dbfs, f.ppm_error = frame.frame_pwr_dbfs, frame.nf_pwr_dbfs, frame.ppm_error
    f.burst_timestamp.tv_sec, f.burst_timestamp.tv_usec = timestamp
    out = (C.c_uint8 * 70000)()
    n = _check(L, L.vdl2gpu_serialize_raw_frame(C.byref(f), station_id.encode() if station_id else None, out, 70000), "vdl2gpu_serialize_raw_frame")
    return bytes(out[:n])


def frame_from_c(f):
    """vdl2gpu_frame (ctypes) -> Frame"""
    o = Frame()
    o.channel, o.freq, o.burst_seq, o.idx = f.channel, f.freq, f.burst_seq, f.idx
    o.data = C.string_at(f.data, f.len) if f.len else b""
    o.synd_weight, o.datalen_octets, o.num_fec_corrections = f.synd_weight, f.datalen_octets, f.num_fec_corrections
    o.frame_pwr_dbfs, o.nf_pwr_dbfs, o.ppm_error = f.frame_pwr_dbfs, f.nf_pwr_dbfs, f.ppm_error
    o.frame_pwr, o.mag_nf = f.frame_pwr, f.mag_nf
    o.sync_dec_index = f.sync_dec_index
    o.burst_timestamp = f.burst_timestamp.tv_sec + 1e-6 * f.burst_timestamp.tv_usec
    o.fcs_ok = bool(f.fcs_ok)
    return o


def make_config(sample_rate, oversample, sample_fmt, centerfreq, freqs, max_ppm=0.0, flags=0):
    """(vdl2gpu_config, the freqs array it points at) for the stage stubs"""
    fr = np.ascontiguousarray(freqs, dtype=np.uint32)
    cfg = _Config()
    cfg.sample_rate, cfg.oversample, cfg.sample_fmt, cfg.centerfreq = sample_rate, oversample, sample_fmt, centerfreq
    cfg.n_channels = int(fr.size)
    cfg.freqs = fr.ctypes.data_as(C.POINTER(C.c_uint32))
    cfg.max_ppm, cfg.flags, cfg.device = max_ppm, flags, -1
    return cfg, fr


def parse_records(region_bytes, decimated_rate):
    """host copy of a vdl2gpu_launch_burst_fec region -> [Frame]"""
    L = load_library()
    out = []
    cb = _FRAME_CB(lambda fp, _u: out.append(frame_from_c(fp.contents)))
    buf = np.frombuffer(region_bytes, np.uint8)
    _check(L, L.vdl2gpu_parse_records(buf.ctypes.data, buf.size, decimated_rate, cb, None), "vdl2gpu_parse_records")
    return out


class Vdl2Channels:
    """N VDL2 channels demodulated from one IQ stream on one B200 (or from many: n_streams, from_streams)."""

    def __init__(self, sample_rate, oversample, sample_fmt, centerfreq, freqs, max_ppm=0.0,
                 max_chunk_bytes=1 << 20, device=-1, flags=0, n_inflight=4, n_streams=1):
        """n_streams > 1: independent-streams mode, channels [s*C, (s+1)*C) demodulate stream s; process_buf_* then take
        the S per-stream buffers back to back."""
        n_streams = int(n_streams)
        self._open(sample_rate, oversample, sample_fmt, centerfreq, freqs, n_streams, None, max_ppm, max_chunk_bytes, device, flags, n_inflight)
        per = self.n_channels // n_streams if n_streams > 1 else self.n_channels
        self.stream_of_channel = np.arange(self.n_channels, dtype=np.int64) // max(per, 1)

    @classmethod
    def from_streams(cls, sample_rate, oversample, sample_fmt, streams, max_ppm=0.0, max_chunk_bytes=1 << 20, device=-1, flags=0,
                     n_inflight=4):
        """Receiver farm (vdl2gpu_create_streams): `streams` is a list of (centerfreq, [freqs...]) pairs, one per receiver;
        a receiver may carry any number of channels, none included.  Channels are numbered stream-major (stream 0's
        first); `stream_of_channel[k]` is channel k's stream.  process_buf_* / submit / submit_device take the
        n_streams per-stream buffers of equal length back to back."""
        streams = list(streams)
        if not streams:
            raise ValueError("from_streams: at least one stream is required")
        centres, counts, freqs = [], [], []
        for k, st in enumerate(streams):
            try:
                centre, fs = st
                fs = [int(f) for f in fs]
            except (TypeError, ValueError):
                raise ValueError(f"from_streams: stream {k} is not a (centerfreq, [freqs...]) pair") from None
            centres.append(int(centre)); counts.append(len(fs)); freqs.extend(fs)
        self = cls.__new__(cls)
        layout = (np.asarray(counts, np.uint32), np.asarray(centres, np.uint32))
        self._open(sample_rate, oversample, sample_fmt, centres[0], freqs, len(streams), layout, max_ppm, max_chunk_bytes, device,
                   flags, n_inflight)
        self.centerfreqs = layout[1]
        self.stream_of_channel = np.repeat(np.arange(len(streams), dtype=np.int64), layout[0])
        return self

    def _open(self, sample_rate, oversample, sample_fmt, centerfreq, freqs, n_streams, layout, max_ppm, max_chunk_bytes, device,
              flags, n_inflight):
        self.L = load_library()
        self.n_streams = int(n_streams)
        self.freqs = np.ascontiguousarray(freqs, dtype=np.uint32)
        self.n_channels = int(self.freqs.size)
        self.sample_fmt = sample_fmt
        cfg = _Config()
        cfg.sample_rate, cfg.oversample, cfg.sample_fmt, cfg.centerfreq = sample_rate, oversample, sample_fmt, centerfreq
        cfg.n_channels = self.n_channels
        cfg.freqs = self.freqs.ctypes.data_as(C.POINTER(C.c_uint32))
        cfg.max_ppm, cfg.max_chunk_bytes, cfg.device, cfg.flags, cfg.n_inflight = max_ppm, max_chunk_bytes, device, flags, n_inflight
        cfg.n_streams = self.n_streams
        self.h = C.c_void_p()
        if layout is None:
            _check(self.L, self.L.vdl2gpu_create(C.byref(cfg), C.byref(self.h)), "vdl2gpu_create")
        else:
            counts, centres = layout
            lay = _StreamLayout(self.n_streams, counts.ctypes.data_as(C.POINTER(C.c_uint32)), centres.ctypes.data_as(C.POINTER(C.c_uint32)))
            _check(self.L, self.L.vdl2gpu_create_streams(C.byref(cfg), C.byref(lay), C.byref(self.h)), "vdl2gpu_create_streams")
        self._frames = []
        self._cb = _FRAME_CB(self._on_frame)

    def close(self):
        if getattr(self, "h", None):
            self.L.vdl2gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _on_frame(self, fp, _user):
        self._frames.append(frame_from_c(fp.contents))

    # ---- the reference's entry points for this path ----
    def process_buf_uchar(self, buf):
        """src/demod.c:339-347: interleaved cu8 I,Q bytes."""
        return self._submit(buf, FMT_U8)

    def process_buf_short(self, buf):
        """src/demod.c:356-365: interleaved little-endian cs16 I,Q."""
        return self._submit(buf, FMT_S16)

    def _submit(self, buf, fmt):
        if fmt != self.sample_fmt:
            raise Vdl2GpuError("sample format differs from the one the channels were created with")
        b = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
        if b.size % self.n_streams:
            raise Vdl2GpuError("buffer size is not a multiple of n_streams")
        _check(self.L, self.L.vdl2gpu_submit(self.h, b.ctypes.data, b.size // self.n_streams), "vdl2gpu_submit")

    def submit(self, buf):
        return self._submit(buf, self.sample_fmt)

    def submit_planar_s16(self, xi, xq):
        """SDRplay-style hand-off: separate int16 I and Q arrays (src/sdrplay.c:72-134)."""
        xi = np.ascontiguousarray(xi, dtype=np.int16); xq = np.ascontiguousarray(xq, dtype=np.int16)
        assert xi.size == xq.size
        _check(self.L, self.L.vdl2gpu_submit_planar_s16(self.h, xi.ctypes.data, xq.ctypes.data, xi.size), "vdl2gpu_submit_planar_s16")

    def submit_device(self, dev_ptr, nbytes, producer_stream=0):
        _check(self.L, self.L.vdl2gpu_submit_device(self.h, C.c_void_p(dev_ptr), nbytes, C.c_void_p(producer_stream)), "vdl2gpu_submit_device")

    def wait_input_consumed(self, stream=0):
        _check(self.L, self.L.vdl2gpu_wait_input_consumed(self.h, C.c_void_p(stream)), "vdl2gpu_wait_input_consumed")

    def stream_wait(self, stream=0):
        _check(self.L, self.L.vdl2gpu_stream_wait(self.h, C.c_void_p(stream)), "vdl2gpu_stream_wait")

    def process_chunked(self, buf, chunk_bytes):
        b = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
        for off in range(0, b.size, chunk_bytes):
            self._submit(b[off:off + chunk_bytes], self.sample_fmt)

    def poll(self):
        """Frames of the chunks finished so far (non-blocking)."""
        _check(self.L, self.L.vdl2gpu_poll(self.h, self._cb, None), "vdl2gpu_poll")
        out, self._frames = self._frames, []
        return out

    def flush(self):
        """Block until everything submitted is processed; returns the frames."""
        _check(self.L, self.L.vdl2gpu_flush(self.h, self._cb, None), "vdl2gpu_flush")
        out, self._frames = self._frames, []
        return out

    def poll_count(self):
        """Like poll() but only counts frames (no Python object per frame)."""
        return _check(self.L, self.L.vdl2gpu_poll(self.h, C.cast(None, _FRAME_CB), None), "vdl2gpu_poll")

    def flush_count(self):
        """Like flush() but only counts frames (no Python object per frame)."""
        return _check(self.L, self.L.vdl2gpu_flush(self.h, C.cast(None, _FRAME_CB), None), "vdl2gpu_flush")

    # ---- introspection ----
    def stats(self):
        s = _Stats()
        _check(self.L, self.L.vdl2gpu_get_stats(self.h, C.byref(s)), "vdl2gpu_get_stats")
        return {n: getattr(s, n) for n, _ in _Stats._fields_ if n != "reserved"}

    def channel_counters(self):
        a = np.zeros((self.n_channels, NUM_COUNTERS), np.uint64)
        _check(self.L, self.L.vdl2gpu_get_channel_counters(self.h, a.ctypes.data, self.n_channels), "vdl2gpu_get_channel_counters")
        return a

    def tables(self):
        t = dict(levels=np.zeros(256, np.float32), sin_lut=np.zeros(257, np.float32), cos_lut=np.zeros(257, np.float32),
                 A=np.zeros(3, np.float32), B=np.zeros(3, np.float32), lr_X=np.zeros(16, np.float32),
                 lr_denom=np.zeros(1, np.float32), pr_phase=np.zeros(16, np.float32))
        _check(self.L, self.L.vdl2gpu_get_tables(self.h, *[t[k].ctypes.data for k in
               ("levels", "sin_lut", "cos_lut", "A", "B", "lr_X", "lr_denom", "pr_phase")]), "vdl2gpu_get_tables")
        return t

    def read_dec(self, max_dec):
        out = np.zeros((max_dec, self.n_channels, 2), np.float32)
        n = C.c_uint32(0)
        _check(self.L, self.L.vdl2gpu_read_dec(self.h, out.ctypes.data, out.size, C.byref(n)), "vdl2gpu_read_dec")
        return out[:n.value]

    def read_events(self, cap=1 << 16):
        ev = (_Event * cap)()
        n = _check(self.L, self.L.vdl2gpu_read_events(self.h, C.cast(ev, C.c_void_p), cap), "vdl2gpu_read_events")
        return [dict(channel=ev[k].channel, kind=ev[k].kind, dec_index=ev[k].dec_index, i=list(ev[k].i),
                     f=np.array(list(ev[k].f), np.float32)) for k in range(n)]

    def enable_timing(self, on=True):
        _check(self.L, self.L.vdl2gpu_enable_timing(self.h, 1 if on else 0), "vdl2gpu_enable_timing")

    def timeline(self, cap=4096):
        """rows of [chunk, front start, K1 end, K2a start, K2a end, K2 start, K2|K3, K3 end] (ms) for the timed chunks"""
        a = np.zeros((cap, 8), np.float32)
        n = _check(self.L, self.L.vdl2gpu_get_timeline(self.h, a.ctypes.data, cap), "vdl2gpu_get_timeline")
        return a[:n]

    def block_trace(self, cap=1 << 16):
        """rows of [kernel, block, smid, 0, start_ns, end_ns] (needs VDL2GPU_BLOCK_TRACE=1 when the object was created)"""
        a = np.zeros((cap, 6), np.uint64)
        n = _check(self.L, self.L.vdl2gpu_debug_block_trace(self.h, a.ctypes.data, cap), "vdl2gpu_debug_block_trace")
        return a[:n]

    def kernel_ms(self):
        ms = (C.c_double * 5)()
        n = (C.c_uint64 * 5)()
        _check(self.L, self.L.vdl2gpu_get_kernel_ms(self.h, ms, n), "vdl2gpu_get_kernel_ms")
        return dict(K0=(ms[0], n[0]), K1=(ms[1], n[1]), K2a=(ms[2], n[2]), K2=(ms[3], n[3]), K3=(ms[4], n[4]))
