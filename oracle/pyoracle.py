"""ctypes binding of oracle/liboracle.so (CPU restatement of the reference hot path).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package (dumpvdl2_b200) must never import this.
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

FMT_U8, FMT_S16 = 0, 1
NUM_COUNTERS = 9
COUNTER_NAMES = ["sync_good", "hdr_crc_good", "bursts", "burst_err", "blocks_processed",
                 "blocks_fec_ok", "msg_good", "fcs_good", "fcs_bad"]


class VoFrame(C.Structure):
    _fields_ = [("channel", C.c_uint32), ("freq", C.c_uint32), ("burst_seq", C.c_uint32),
                ("idx", C.c_int32), ("len", C.c_uint32), ("offset", C.c_uint32),
                ("synd_weight", C.c_uint32), ("datalen_octets", C.c_uint32),
                ("num_fec_corrections", C.c_int32), ("frame_pwr", C.c_float), ("mag_nf", C.c_float),
                ("frame_pwr_dbfs", C.c_float), ("nf_pwr_dbfs", C.c_float), ("ppm_error", C.c_float),
                ("sync_dec_index", C.c_uint64), ("fcs_residue", C.c_uint16), ("pad", C.c_uint16)]


class VoEvent(C.Structure):
    _fields_ = [("channel", C.c_uint32), ("kind", C.c_uint32), ("dec_index", C.c_uint64),
                ("i", C.c_int32 * 8), ("f", C.c_float * 8)]


def build(force=False):
    """(Re)build liboracle.so and, when the reference sources are present (REF in oracle/Makefile), oracle/_ref."""
    so = os.path.join(_HERE, "liboracle.so")
    src = [os.path.join(_HERE, f) for f in ("vdl2_oracle.c", "vdl2_oracle.h")]
    stale = force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src)
    if stale:
        subprocess.check_call(["make", "-C", _HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", _HERE, "ref"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    so = build()
    L = C.CDLL(so)
    L.vo_create.restype = C.c_void_p
    L.vo_create.argtypes = [C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32, C.c_float]
    L.vo_destroy.argtypes = [C.c_void_p]
    L.vo_process.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.vo_num_frames.restype = C.c_uint32
    L.vo_num_frames.argtypes = [C.c_void_p]
    L.vo_frames.restype = C.POINTER(VoFrame)
    L.vo_frames.argtypes = [C.c_void_p]
    L.vo_frame_bytes.restype = C.POINTER(C.c_uint8)
    L.vo_frame_bytes.argtypes = [C.c_void_p]
    L.vo_enable_trace.argtypes = [C.c_void_p, C.c_int]
    L.vo_num_events.restype = C.c_uint32
    L.vo_num_events.argtypes = [C.c_void_p]
    L.vo_events.restype = C.POINTER(VoEvent)
    L.vo_events.argtypes = [C.c_void_p]
    L.vo_enable_dec_tap.argtypes = [C.c_void_p, C.c_int]
    L.vo_dec_count.restype = C.c_uint64
    L.vo_dec_count.argtypes = [C.c_void_p]
    L.vo_dec_tap.restype = C.POINTER(C.c_float)
    L.vo_dec_tap.argtypes = [C.c_void_p]
    L.vo_counters.restype = C.POINTER(C.c_uint64)
    L.vo_counters.argtypes = [C.c_void_p]
    L.vo_levels_u8.argtypes = [C.c_void_p]
    L.vo_sincos_lut.argtypes = [C.c_void_p, C.c_void_p]
    L.vo_lpf_design.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p]
    L.vo_sync_consts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.vo_downmix_dphi.restype = C.c_uint32
    L.vo_downmix_dphi.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32]
    L.vo_header_decode.restype = C.c_uint32
    L.vo_header_decode.argtypes = [C.POINTER(C.c_uint32)]
    L.vo_header_encode.restype = C.c_uint32
    L.vo_header_encode.argtypes = [C.c_uint32]
    L.vo_synd_weight.restype = C.c_uint32
    L.vo_synd_weight.argtypes = [C.c_uint32]
    L.vo_reverse_bits.restype = C.c_uint32
    L.vo_reverse_bits.argtypes = [C.c_uint32, C.c_int]
    L.vo_fec_octets_for.restype = C.c_int
    L.vo_fec_octets_for.argtypes = [C.c_uint32]
    L.vo_rs_verify.restype = C.c_int
    L.vo_rs_verify.argtypes = [C.c_void_p, C.c_int]
    L.vo_rs_encode.argtypes = [C.c_void_p]
    L.vo_crc16.restype = C.c_uint16
    L.vo_crc16.argtypes = [C.c_void_p, C.c_uint32, C.c_uint16]
    L.vo_scramble_bits.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint16)]
    L.vo_decode_burst_bits.restype = C.c_int
    L.vo_decode_burst_bits.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_int32), C.c_void_p]
    _LIB = L
    return L


class Frame:
    """One AVLC frame + metadata, the unit compared between implementations."""
    __slots__ = ("channel", "freq", "burst_seq", "idx", "data", "synd_weight", "datalen_octets",
                 "num_fec_corrections", "frame_pwr", "mag_nf", "frame_pwr_dbfs", "nf_pwr_dbfs",
                 "ppm_error", "sync_dec_index", "fcs_ok")

    def key(self):
        return (self.channel, self.burst_seq, self.idx)

    def __repr__(self):
        return (f"Frame(ch={self.channel} burst={self.burst_seq} idx={self.idx} len={len(self.data)} "
                f"fcs_ok={self.fcs_ok} fec={self.num_fec_corrections} synd={self.synd_weight})")


class Oracle:
    """Whole-path oracle for one IQ stream fanned out to n channels."""

    def __init__(self, sample_rate, oversample, fmt, centerfreq, freqs, max_ppm=0.0, trace=False, dec_tap=False):
        self.L = lib()
        self.freqs = np.ascontiguousarray(freqs, dtype=np.uint32)
        self.n_channels = len(self.freqs)
        self.fmt = fmt
        self.h = self.L.vo_create(sample_rate, oversample, fmt, centerfreq,
                                  self.freqs.ctypes.data_as(C.POINTER(C.c_uint32)), self.n_channels, max_ppm)
        if trace:
            self.L.vo_enable_trace(self.h, 1)
        if dec_tap:
            self.L.vo_enable_dec_tap(self.h, 1)

    def close(self):
        if self.h:
            self.L.vo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def process(self, buf):
        b = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
        self.L.vo_process(self.h, b.ctypes.data, b.size)

    def process_chunked(self, buf, chunk_bytes):
        b = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
        for off in range(0, b.size, chunk_bytes):
            part = b[off:off + chunk_bytes]
            self.L.vo_process(self.h, part.ctypes.data, part.size)

    def frames(self):
        n = self.L.vo_num_frames(self.h)
        fr = self.L.vo_frames(self.h)
        arena = self.L.vo_frame_bytes(self.h)
        out = []
        for k in range(n):
            f = fr[k]
            o = Frame()
            o.channel, o.freq, o.burst_seq, o.idx = f.channel, f.freq, f.burst_seq, f.idx
            o.data = bytes(bytearray(arena[f.offset:f.offset + f.len])) if f.len else b""
            o.synd_weight, o.datalen_octets = f.synd_weight, f.datalen_octets
            o.num_fec_corrections = f.num_fec_corrections
            o.frame_pwr, o.mag_nf = f.frame_pwr, f.mag_nf
            o.frame_pwr_dbfs, o.nf_pwr_dbfs, o.ppm_error = f.frame_pwr_dbfs, f.nf_pwr_dbfs, f.ppm_error
            o.sync_dec_index = f.sync_dec_index
            o.fcs_ok = (f.fcs_residue == 0xF0B8) and f.len >= 11
            out.append(o)
        return out

    def events(self):
        n = self.L.vo_num_events(self.h)
        ev = self.L.vo_events(self.h)
        return [dict(channel=ev[k].channel, kind=ev[k].kind, dec_index=ev[k].dec_index,
                     i=list(ev[k].i), f=np.array(list(ev[k].f), dtype=np.float32)) for k in range(n)]

    def dec_samples(self):
        n = self.L.vo_dec_count(self.h)
        if n == 0:
            return np.zeros((0, self.n_channels, 2), np.float32)
        p = self.L.vo_dec_tap(self.h)
        return np.ctypeslib.as_array(p, shape=(n, self.n_channels, 2)).copy()

    def counters(self):
        p = self.L.vo_counters(self.h)
        return np.ctypeslib.as_array(p, shape=(self.n_channels, NUM_COUNTERS)).copy()


# ---- stage-level helpers ----
def levels_u8():
    a = np.zeros(256, np.float32); lib().vo_levels_u8(a.ctypes.data); return a


def sincos_lut():
    s = np.zeros(257, np.float32); c = np.zeros(257, np.float32)
    lib().vo_sincos_lut(s.ctypes.data, c.ctypes.data); return s, c


def lpf_design(rate):
    a = np.zeros(3, np.float32); b = np.zeros(3, np.float32)
    lib().vo_lpf_design(rate, a.ctypes.data, b.ctypes.data); return a, b


def sync_consts():
    x = np.zeros(16, np.float32); d = np.zeros(1, np.float32); p = np.zeros(16, np.float32)
    lib().vo_sync_consts(x.ctypes.data, d.ctypes.data, p.ctypes.data); return x, float(d[0]), p


def rs_encode(block249):
    b = np.zeros(255, np.uint8); b[:249] = np.frombuffer(bytes(block249), np.uint8)
    lib().vo_rs_encode(b.ctypes.data); return b


def rs_verify(block255, fec_octets):
    b = np.array(block255, dtype=np.uint8).copy()
    r = lib().vo_rs_verify(b.ctypes.data, fec_octets); return r, b


def crc16(data, init=0xFFFF):
    b = np.frombuffer(bytes(data), np.uint8)
    return lib().vo_crc16(b.ctypes.data if b.size else None, b.size, init)


def scramble(bits, lfsr=0x6959):
    b = np.array(bits, dtype=np.uint8).copy()
    st = C.c_uint16(lfsr)
    lib().vo_scramble_bits(b.ctypes.data, b.size, C.byref(st))
    return b, st.value


def decode_burst_bits(bits, datalen_bits):
    b = np.ascontiguousarray(bits, dtype=np.uint8)
    out = np.zeros(4096, np.uint8); lens = np.zeros(1100, np.uint32)
    n = C.c_uint32(0); corr = C.c_int32(0); rs = np.zeros(9, np.int8)
    st = lib().vo_decode_burst_bits(b.ctypes.data, b.size, datalen_bits, out.ctypes.data, out.size,
                                    lens.ctypes.data, lens.size, C.byref(n), C.byref(corr), rs.ctypes.data)
    frames, off = [], 0
    for k in range(n.value):
        frames.append(bytes(out[off:off + lens[k]])); off += int(lens[k])
    return st, frames, corr.value, rs


# ---- the unmodified reference, when oracle/_ref was built (this container, or shipped prebuilt) ----
def ref_binary(flavour="strict"):
    p = os.path.join(_HERE, "_ref", f"vdl2_ref_{flavour}")
    return p if os.path.exists(p) else None


def run_ref(path, fmt, oversample, centerfreq, freqs, flavour="strict", chunk=None, loop=1, quiet=False, max_ppm=None, pin=False):
    """Run oracle/_ref/vdl2_ref_<flavour> on an IQ file; returns (frames as dicts, stats dict)."""
    exe = ref_binary(flavour)
    if exe is None:
        raise FileNotFoundError("oracle/_ref not built")
    cmd = [exe, "--fmt", "s16" if fmt == FMT_S16 else "u8", "--oversample", str(oversample),
           "--centerfreq", str(centerfreq), "--freqs", ",".join(str(int(f)) for f in freqs), "--loop", str(loop)]
    if chunk:
        cmd += ["--chunk", str(chunk)]
    if max_ppm:
        cmd += ["--max-ppm", str(max_ppm)]
    if quiet:
        cmd += ["--quiet"]
    if pin:
        cmd += ["--pin"]
    cmd.append(path)
    out = subprocess.run(cmd, check=True, capture_output=True, text=True).stdout
    frames, stats = [], {}
    for line in out.splitlines():
        kv = dict(t.split("=", 1) for t in line.split()[1:])
        if line.startswith("FRAME"):
            frames.append(dict(channel=int(kv["ch"]), freq=int(kv["freq"]), idx=int(kv["idx"]),
                               data=bytes.fromhex(kv.get("hex", "")), synd_weight=int(kv["synd"]),
                               datalen_octets=int(kv["datalen"]), num_fec_corrections=int(kv["fec"]),
                               frame_pwr_dbfs=float(kv["pwr"]), nf_pwr_dbfs=float(kv["nf"]), ppm_error=float(kv["ppm"])))
        elif line.startswith("STATS"):
            stats = {k: float(v) for k, v in kv.items()}
    return frames, stats
