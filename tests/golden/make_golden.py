"""Generate tests/golden/*.json by running the UNMODIFIED reference (oracle/_ref/vdl2_ref_{strict,fast},
built from the reference sources by oracle/Makefile) on the deterministic streams of tests/cases.py, and by
reading the reference's table literals and struct layout.  Needs a dumpvdl2 source tree:

    python tests/golden/make_golden.py /path/to/dumpvdl2
"""
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np
from oracle import pyoracle as po
from tests import cases


def write(name, obj):
    with open(os.path.join(cases.GOLDEN, f"{name}.json"), "w") as f:
        json.dump(obj, f, indent=1)


def ref_tables(ref):
    """header FEC parity rows, syndrome table, syndrome weights and CRC-16 table as the reference spells them (src/decode.c, src/crc.c)"""
    src = open(os.path.join(ref, "src", "decode.c")).read()
    rows = [int(x, 2) for x in re.findall(r"0b([01]{25})", src.split("syndtable")[0])]
    pats = [int(x, 2) for x in re.findall(r"0b([01]{25})", src.split("syndtable")[1].split("synd_weight")[0])]
    weights = [int(x) for x in re.findall(r"\d+", src.split("synd_weight[1<<HDRFECLEN] = {")[1].split("}")[0])]
    crc = [int(x, 16) for x in re.findall(r"0x([0-9A-F]{4})", open(os.path.join(ref, "src", "crc.c")).read().split("crctable[256]")[1])][:256]
    return dict(syndrome_rows=rows, syndrome_patterns=pats, synd_weight=weights, crc16_table=crc)


def ref_layout():
    """sizes and offsets of the reference structs the drop-in mirrors (oracle/layout_check.c, x86-64)"""
    out = subprocess.run([os.path.join(ROOT, "oracle", "_ref", "layout_check")], capture_output=True, text=True).stdout
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"^(\S+(?: \S+)?)\s+reference\s+(\d+)", out, re.M)}


def main():
    ref = os.path.abspath(sys.argv[1])
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), f"REF={ref}", "ref"], stdout=subprocess.DEVNULL)
    for name, fn in {**cases.ALL_GOLDEN, **cases.ORACLE_GOLDEN}.items():
        c = fn()
        with tempfile.NamedTemporaryFile(suffix=".iq", delete=False) as tf:
            if name == "wav":
                tf.write(c["raw_bytes"])      # the reference feeds the whole file, header included
            else:
                tf.write(np.ascontiguousarray(c["iq"]).view(np.uint8).tobytes())
            path = tf.name
        out = dict(name=name, fs=c["fs"], oversample=c["oversample"], fmt=c["fmt"], centerfreq=c["centerfreq"],
                   freqs=c["freqs"], chunk=c["chunk"], iq_sha256=cases.iq_sha256(c),
                   injected=[[f.hex() for f in b.frames] for b in c["bursts"]])
        for fl in ("strict", "fast"):
            fr, _ = po.run_ref(path, po.FMT_S16 if c["fmt"] == "s16" else po.FMT_U8, c["oversample"], c["centerfreq"],
                               c["freqs"], flavour=fl, chunk=c["chunk"])
            out[fl] = [dict(channel=f["channel"], idx=f["idx"], hex=f["data"].hex(), synd_weight=f["synd_weight"],
                            datalen_octets=f["datalen_octets"], num_fec_corrections=f["num_fec_corrections"],
                            frame_pwr_dbfs=f["frame_pwr_dbfs"], nf_pwr_dbfs=f["nf_pwr_dbfs"], ppm_error=f["ppm_error"]) for f in fr]
        os.unlink(path)
        write(name, out)
        same = [x["hex"] for x in out["strict"]] == [x["hex"] for x in out["fast"]]
        ninj = sum(len(b) for b in out["injected"])
        print(f"{name}: strict {len(out['strict'])} frames, fast {len(out['fast'])} frames, injected {ninj}, strict==fast bytes: {same}")
    write("ref_tables", ref_tables(ref))
    write("dropin_layout", ref_layout())


if __name__ == "__main__":
    main()
