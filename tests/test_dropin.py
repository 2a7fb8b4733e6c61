"""The drop-in boundary: the reference's own init/feed protocol (oracle/dropin_harness.c = what src/dumpvdl2.c does:
vdl2_channel_init xN, rs_init, ..., barriers, one process_samples pthread per channel, process_buf_* per chunk,
final demods_ready wait) linked against libvdl2gpu.so instead of src/demod.c + src/rs.c + src/libfec, with the
frames captured where the reference's src/decode.c receives them (avlc_decoder_queue_push).  Output must equal the
unmodified reference's, stored in tests/golden."""
import os
import subprocess
import tempfile
import pytest
from tests import cases, util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "dumpvdl2_b200")


def _cc(tmp, src, out, *extra):
    exe = str(tmp / out)
    subprocess.check_call(["gcc", "-O2", "-std=c11", "-D_DEFAULT_SOURCE", "-pthread", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "oracle", src), "-o", exe, *extra])
    return exe


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    return _cc(tmp_path_factory.mktemp("dropin"), "dropin_harness.c", "dropin_harness",
               "-L", LIBDIR, "-lvdl2gpu", "-Wl,-rpath," + LIBDIR)


def test_layout_mirrors_match_reference_headers(tmp_path):
    """the layout mirrors of include/vdl2_dropin.h against the reference's own declarations (src/dumpvdl2.h:321-352,
    422-425, src/output-common.h:31-43), whose sizes and offsets tests/golden/dropin_layout.json stores"""
    want = util.load_golden("dropin_layout")
    out = subprocess.run([_cc(tmp_path, "layout_mirror.c", "layout_mirror")], capture_output=True, text=True, check=True).stdout
    got = dict(line.split("\t") for line in out.splitlines())
    assert len(want) >= 10 and sorted(got) == sorted(want)
    for k, v in want.items():
        assert int(got[k]) == v, f"{k}: mirror {got[k]}, reference {v}"


def test_harness_links_against_the_product_library(harness):
    out = subprocess.run(["ldd", harness], capture_output=True, text=True).stdout
    assert "libvdl2gpu.so" in out and "not found" not in out.split("libvdl2gpu.so")[1].splitlines()[0]


def _run_harness(harness, case):
    with tempfile.NamedTemporaryFile(suffix=".iq", delete=False) as tf:
        tf.write(util.case_bytes(case).tobytes())
        path = tf.name
    try:
        cmd = [harness, "--fmt", "s16" if case["fmt"] == "s16" else "u8", "--oversample", str(case["oversample"]),
               "--centerfreq", str(case["centerfreq"]), "--freqs", ",".join(str(f) for f in case["freqs"]),
               "--chunk", str(case["chunk"]), path]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        frames = []
        for line in r.stdout.splitlines():
            if line.startswith("FRAME"):
                frames.append(dict(t.split("=", 1) for t in line.split()[1:]))
        return frames
    finally:
        os.unlink(path)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["wav", "cfg2", "mixed_s16"])
def test_dropin_harness_reproduces_reference_output(name, harness):
    c = cases.ALL_GOLDEN[name]()
    got = _run_harness(harness, c)
    want = util.load_golden(name)["strict"]
    assert len(got) == len(want)
    for a, b in zip(got, want):          # same print order: per channel, push order
        assert int(a["ch"]) == b["channel"] and int(a["idx"]) == b["idx"] and a.get("hex", "") == b["hex"]
        assert int(a["synd"]) == b["synd_weight"] and int(a["datalen"]) == b["datalen_octets"] and int(a["fec"]) == b["num_fec_corrections"]
        for k, g in (("pwr", "frame_pwr_dbfs"), ("nf", "nf_pwr_dbfs"), ("ppm", "ppm_error")):
            assert float(a[k]) == float(f"{b[g]:.9g}"), (k, a[k], b[g])
