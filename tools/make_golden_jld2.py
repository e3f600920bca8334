"""Writes tests/golden/jld2_results.npz: the reference's LotkaVolterra/results/*.jld2 files that tests/test_jld2_reader.py reads,
shrunk so that the suite does not need the reference checkout.  Every byte the JLD2 reader visits is kept verbatim: the text header
and superblock, the object headers (with their continuation blocks and checksums) of every root link, the data of every plain numeric
dataset, and the records and objects `read_tree` reaches from the parameter containers.  Every other byte is zeroed and the file keeps
its length, so addresses, checksums and the reader's results are those of the original file; the zeros compress away.
    python tools/make_golden_jld2.py --ref <checkout of the reference>"""
import argparse
import hashlib
import os
import struct
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from universal_differential_equations_b200 import jld2  # noqa: E402

FILES = {"hudson_bay": "Hudson_Bay_recovery.jld2", "scenario_1": "Scenario_1_recovery_0.005.jld2",
         "scenario_2": "Scenario_2_recovery_0.005.jld2", "scenario_3": "Scenario_3_recovery_0.005.jld2"}   # under LotkaVolterra/results
FOLLOW = ("trained_parameters", "initial_parameters")     # the parameter containers whose references read_tree follows


def header_ranges(f, addr):
    """Byte ranges of the object header at addr: its first chunk with the checksum and every continuation block."""
    b, pos = f.blob, f.base + addr
    flags = b[pos + 5]
    q = pos + 6 + (16 if flags & 0x20 else 0) + (4 if flags & 0x10 else 0)
    n = 1 << (flags & 3)
    out = [(pos, q + n + int.from_bytes(b[q:q + n], "little") + 4)]
    blocks, tracked = [(q + n, out[0][1] - 4)], bool(flags & 0x04)     # the message walk of JLD2File._messages, continuations included
    while blocks:
        p, end = blocks.pop(0)
        while p + 4 <= end:
            mtype, msize = b[p], struct.unpack_from("<H", b, p + 1)[0]
            p += 4 + (2 if tracked else 0)
            if mtype == 0x10:
                off, length = struct.unpack_from("<QQ", b, p)
                out.append((f.base + off, f.base + off + length))
                blocks.append((f.base + off + 4, f.base + off + length - 4))
            p += msize
    return out


def object_ranges(f, addr, follow, depth=0):
    """Header ranges of the object at addr, its contiguous data, and (follow) what read_tree reaches from it."""
    out = header_ranges(f, addr)
    dims, dtype, layout = f._describe_at(addr)
    if layout is not None and layout[0] == "contiguous" and layout[1] != jld2.UNDEF and (follow or dtype is not None):
        out.append((f.base + layout[1], f.base + layout[1] + layout[2]))
    if follow and not (dims is not None and dtype is not None) and layout is not None and depth < 8:
        raw = layout[1] if layout[0] == "compact" else f.blob[f.base + layout[1]:f.base + layout[1] + layout[2]]
        for k in range(0, len(raw) - 7, 8):
            ref = struct.unpack_from("<Q", raw, k)[0]
            if f._object_at(ref):
                out += object_ranges(f, ref, True, depth + 1)
    return out


def shrink(path):
    f = jld2.JLD2File(path)
    sb = f.blob.find(jld2._SIG)
    keep = [(0, sb + 48)] + header_ranges(f, struct.unpack_from("<Q", f.blob, sb + 36)[0])    # text header, superblock, root group
    for name, addr in f.links.items():
        keep += object_ranges(f, addr, name in FOLLOW)
    out = bytearray(len(f.blob))
    for lo, hi in keep:
        out[lo:hi] = f.blob[lo:hi]
    return bytes(out)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", required=True, help="checkout of ChrisRackauckas/universal_differential_equations")
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "jld2_results.npz"))
    a = ap.parse_args()
    arrays = {}
    for key, fn in FILES.items():
        path = os.path.join(a.ref, "LotkaVolterra", "results", fn)
        blob, small = open(path, "rb").read(), shrink(path)
        arrays[key] = np.frombuffer(small, np.uint8)
        arrays[key + "_source"] = np.array(f"LotkaVolterra/results/{fn} sha256={hashlib.sha256(blob).hexdigest()}")
        kept = sum(1 for x, y in zip(small, blob) if x == y and x)
        print(f"{key}: {fn}, {len(blob)} bytes, {kept} non-zero bytes kept, deflated {len(zlib.compress(small, 9))} bytes")
    np.savez_compressed(a.out, **arrays)
    print("wrote", a.out, os.path.getsize(a.out), "bytes")
