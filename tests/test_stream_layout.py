"""CPU: receiver-farm contexts (vdl2gpu_create_streams, Vdl2Channels.from_streams).  A malformed layout is refused with
VDL2GPU_EINVAL before any device call, so these run without a GPU; a valid one reaches the device probe."""
import ctypes as C
import numpy as np
import pytest
import dumpvdl2_b200 as vd
from dumpvdl2_b200 import api

EINVAL, ENODEV = -1, -2
CENTER = 136975000


def _gpu_present():
    import torch
    return torch.cuda.is_available()


def _create(counts=(2, 0, 1), centres=(CENTER, CENTER + 4000000, CENTER - 3000000), freqs=None, oversample=20, fmt=vd.FMT_U8,
            flags=0, cfg_streams=0, layout=True, null_counts=False):
    """vdl2gpu_create_streams on a 3-stream layout (2, 0 and 1 channels) -> (return code, last error text)"""
    L = vd.load_library()
    if freqs is None:
        freqs = [centres[0] + 25000, centres[0] - 50000, centres[2] + 100000]
    fr = np.asarray(freqs, np.uint32)
    cn = np.asarray(counts, np.uint32)
    ce = None if centres is None else np.asarray(centres, np.uint32)
    cfg = api._Config()
    cfg.sample_rate, cfg.oversample, cfg.sample_fmt, cfg.centerfreq = 105000 * oversample, oversample, fmt, CENTER
    cfg.n_channels, cfg.freqs = fr.size, fr.ctypes.data_as(C.POINTER(C.c_uint32))
    cfg.flags, cfg.n_streams, cfg.device = flags, cfg_streams, -1
    lay = api._StreamLayout(len(counts), None if null_counts else cn.ctypes.data_as(C.POINTER(C.c_uint32)),
                            None if ce is None else ce.ctypes.data_as(C.POINTER(C.c_uint32)))
    h = C.c_void_p()
    rc = L.vdl2gpu_create_streams(C.byref(cfg), C.byref(lay) if layout else None, C.byref(h))
    if rc == 0:
        L.vdl2gpu_destroy(h)
    return rc, L.vdl2gpu_last_error().decode()


@pytest.mark.parametrize("kw, text", [
    (dict(layout=False), "layout"),
    (dict(null_counts=True), "channels_per_stream"),
    (dict(counts=(2, 0, 2)), "sums to 4"),
    (dict(counts=(1, 0, 1)), "sums to 2"),
    (dict(cfg_streams=2), "cfg->n_streams"),
    (dict(freqs=[CENTER + 25000, CENTER + 1050000, CENTER - 3000000]), "channel 1"),     # exactly sample_rate/2 away
    (dict(freqs=[CENTER + 25000, CENTER - 50000, CENTER + 100000]), "channel 2"),         # beyond: stream 2 is at -3 MHz
    (dict(centres=None, freqs=[CENTER, CENTER, CENTER + 2000000]), "channel 2"),          # NULL centres: cfg->centerfreq
    (dict(oversample=16), "oversample"),
    (dict(oversample=8), "oversample"),
    (dict(fmt=2), "bad vdl2gpu_config"),
    (dict(flags=vd.FLAG_K1_SCALAR), "K1_SCALAR"),
])
def test_malformed_layout_is_refused_before_any_device_call(kw, text):
    rc, err = _create(**kw)
    assert rc == EINVAL, (rc, err)
    assert text in err


def test_zero_streams_and_null_config_are_refused():
    L = vd.load_library()
    h = C.c_void_p()
    lay = api._StreamLayout(0, None, None)
    assert L.vdl2gpu_create_streams(None, C.byref(lay), C.byref(h)) == EINVAL
    rc, err = _create(counts=(), centres=(), freqs=[CENTER])
    assert rc == EINVAL and "n_streams >= 1" in err


@pytest.mark.parametrize("kw", [dict(), dict(cfg_streams=3), dict(oversample=10, fmt=vd.FMT_S16), dict(oversample=13),
                                dict(centres=None, freqs=[CENTER + 25000, CENTER, CENTER - 1000000])])
def test_valid_layout_reaches_the_device_probe(kw):
    if _gpu_present():
        pytest.skip("a GPU is present")
    rc, err = _create(**kw)
    assert rc == ENODEV, (rc, err)


def test_from_streams_argument_handling():
    for bad in ([], [(CENTER,)], [(CENTER, [CENTER], 3)], [CENTER], [(CENTER, ["x"])]):
        with pytest.raises(ValueError):
            vd.Vdl2Channels.from_streams(2100000, 20, vd.FMT_U8, bad)
    # the second channel lies 5 MHz from stream 0's centre but 25 kHz from its own: accepted only if the per-stream
    # centres reach the library
    far = CENTER + 5000000
    if not _gpu_present():
        with pytest.raises(vd.Vdl2GpuError, match="no usable CUDA device"):
            vd.Vdl2Channels.from_streams(2100000, 20, vd.FMT_U8, [(CENTER, [CENTER + 25000]), (far, []), (far, [far + 25000])])
    with pytest.raises(vd.Vdl2GpuError, match="invalid argument"):
        vd.Vdl2Channels.from_streams(2100000, 20, vd.FMT_U8, [(CENTER, [CENTER + 25000]), (CENTER, [far + 25000])])
    with pytest.raises(vd.Vdl2GpuError, match="invalid argument"):
        vd.Vdl2Channels.from_streams(2100000, 20, vd.FMT_U8, [(CENTER, [CENTER + 25000])], flags=vd.FLAG_K1_SCALAR)


def test_header_declares_the_layout_struct_as_ctypes_mirrors_it():
    assert C.sizeof(api._StreamLayout) == 24
    assert [n for n, _ in api._StreamLayout._fields_] == ["n_streams", "channels_per_stream", "centerfreqs"]
    assert api._StreamLayout.channels_per_stream.offset == 8 and api._StreamLayout.centerfreqs.offset == 16
