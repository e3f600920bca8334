"""Reader and writer for the plain numeric datasets of the JLD2 files the reference's scripts write and read
(`save(joinpath(pwd(), "results", "....jld2"), "X", Xn, "t", ts, "losses", losses, ...)`, LotkaVolterra/scenario_1.jl:210-213,
hudson_bay.jl:231-235) -- the data format either side of the training path (SURVEY.md section 8 f4).

JLD2 0.1.x is an HDF5 container behind a 512-byte text header: superblock version 2, version-2 object headers ("OHDR", continued in
"OCHK" blocks), hard links in link messages.  This module walks the root group's links -- and, for slash paths such as "17/X", the
link messages of the groups on the way (`JLD2.Group`, loop_recoveries.jl's one group per run) -- and decodes the datasets whose element type is an
IEEE float or an integer with contiguous or compact layout -- the arrays a training run needs (data X, time points t, loss histories).
Julia structs (the `ODESolution`, `ComponentVector`, Lux chains ... that the same files hold as committed compound types with object
references) are listed by `keys()`; `read_tree` follows a parameter container's references to its arrays, nothing else of a struct is
decoded.  `save` writes Float32 / Float64 arrays with exactly the messages JLD2 itself emits
for them (fill value, version-2 dataspace, IEEE datatype, compact or contiguous layout, lookup3 checksums): the dataset object headers
it produces for the reference's own X / t / losses arrays are byte-identical to the ones in the reference's files (tests/test_jld2_reader.py).
Pure Python + numpy, host side only; no HDF5 library is needed or used.
"""
import struct

import numpy as np

_SIG = b"\x89HDF\r\n\x1a\n"
UNDEF = 0xFFFFFFFFFFFFFFFF
COMPACT_BELOW = 8192          # bytes: smaller arrays are stored inside the object header (what the reference's files show)


def _rot(x, k):
    return ((x << k) | (x >> (32 - k))) & 0xFFFFFFFF


def lookup3(data, init=0):
    """Bob Jenkins' lookup3 `hashlittle`: the checksum of HDF5 version-2 superblocks and object headers."""
    M = 0xFFFFFFFF
    a = b = c = (0xDEADBEEF + len(data) + init) & M
    n, p = len(data), 0
    while n > 12:
        a = (a + int.from_bytes(data[p:p + 4], "little")) & M
        b = (b + int.from_bytes(data[p + 4:p + 8], "little")) & M
        c = (c + int.from_bytes(data[p + 8:p + 12], "little")) & M
        a = (a - c) & M; a ^= _rot(c, 4); c = (c + b) & M
        b = (b - a) & M; b ^= _rot(a, 6); a = (a + c) & M
        c = (c - b) & M; c ^= _rot(b, 8); b = (b + a) & M
        a = (a - c) & M; a ^= _rot(c, 16); c = (c + b) & M
        b = (b - a) & M; b ^= _rot(a, 19); a = (a + c) & M
        c = (c - b) & M; c ^= _rot(b, 4); b = (b + a) & M
        p += 12; n -= 12
    if n == 0:
        return c
    t = bytes(data[p:]) + b"\0" * (12 - n)
    a = (a + int.from_bytes(t[0:4], "little")) & M
    b = (b + int.from_bytes(t[4:8], "little")) & M
    c = (c + int.from_bytes(t[8:12], "little")) & M
    c ^= b; c = (c - _rot(b, 14)) & M
    a ^= c; a = (a - _rot(c, 11)) & M
    b ^= a; b = (b - _rot(a, 25)) & M
    c ^= b; c = (c - _rot(b, 16)) & M
    a ^= c; a = (a - _rot(c, 4)) & M
    b ^= a; b = (b - _rot(a, 14)) & M
    c ^= b; c = (c - _rot(b, 24)) & M
    return c


class JLD2File:
    def __init__(self, path):
        self.blob = open(path, "rb").read()
        b = self.blob
        if not b.startswith(b"HDF5-based Julia Data Format"):
            raise ValueError(f"{path}: not a JLD2 file")
        i = b.find(_SIG)
        if i < 0 or b[i + 8] not in (2, 3) or b[i + 9] != 8 or b[i + 10] != 8:
            raise ValueError(f"{path}: unsupported HDF5 superblock (need version 2 / 3 with 8-byte offsets and lengths)")
        self.base, _ext, _eof, root = struct.unpack_from("<QQQQ", b, i + 12)
        self.superblock_ok = lookup3(b[i:i + 44]) == struct.unpack_from("<I", b, i + 44)[0]
        self.links = self._group_links(root)

    def _group_links(self, addr):
        """{name: object address} of the hard links in the link messages of the group object at addr."""
        links = {}
        for mtype, data in self._messages(addr):
            if mtype == 6:
                name, target = self._link(data)
                if target is not None:
                    links[name] = target
        return links

    def _addr(self, path):
        """Object address of a root link or of a slash path through groups ("17/X"); KeyError when a component is missing."""
        parts = [p for p in path.split("/") if p]
        if not parts:
            raise KeyError(path)
        links = self.links
        for i, part in enumerate(parts):
            if part not in links:
                raise KeyError(path)
            if i == len(parts) - 1:
                return links[part]
            links = self._group_links(links[part])

    # ---- object headers (version 2) ----
    def _messages(self, addr):
        b, pos = self.blob, self.base + addr
        if b[pos:pos + 4] != b"OHDR" or b[pos + 4] != 2:
            raise ValueError("unsupported object header (need version 2)")
        flags = b[pos + 5]
        pos += 6
        if flags & 0x20:
            pos += 16
        if flags & 0x10:
            pos += 4
        n = 1 << (flags & 3)
        size = int.from_bytes(b[pos:pos + n], "little")
        pos += n
        blocks = [(pos, pos + size)]
        tracked = bool(flags & 0x04)
        while blocks:
            p, end = blocks.pop(0)
            while p + 4 <= end:
                mtype = b[p]
                msize = struct.unpack_from("<H", b, p + 1)[0]
                p += 4 + (2 if tracked else 0)
                data = b[p:p + msize]
                p += msize
                if mtype == 0x10:                       # continuation: another block of messages ("OCHK" ... checksum)
                    off, length = struct.unpack_from("<QQ", data, 0)
                    q = self.base + off
                    if b[q:q + 4] != b"OCHK":
                        raise ValueError("bad object header continuation")
                    blocks.append((q + 4, q + length - 4))
                elif mtype != 0:
                    yield mtype, data

    @staticmethod
    def _link(d):
        flags = d[1]
        p = 2
        ltype = 0
        if flags & 0x08:
            ltype = d[p]; p += 1
        if flags & 0x04:
            p += 8
        if flags & 0x10:
            p += 1
        n = 1 << (flags & 3)
        ln = int.from_bytes(d[p:p + n], "little"); p += n
        name = d[p:p + ln].decode("utf-8"); p += ln
        return name, (struct.unpack_from("<Q", d, p)[0] if ltype == 0 else None)

    def header_bytes(self, name):
        """(bytes of the first chunk of the named object's header including its checksum, checksum valid?)"""
        b, pos = self.blob, self.base + self._addr(name)
        flags = b[pos + 5]
        q = pos + 6 + (16 if flags & 0x20 else 0) + (4 if flags & 0x10 else 0)
        n = 1 << (flags & 3)
        end = q + n + int.from_bytes(b[q:q + n], "little")
        return b[pos:end + 4], lookup3(b[pos:end]) == struct.unpack_from("<I", b, end)[0]

    # ---- datasets ----
    def keys(self, group=None):
        """Names of the root links, or of the links of the group at the slash path `group`."""
        return list(self.links if group is None else self._group_links(self._addr(group)))

    def _describe(self, name):
        return self._describe_at(self._addr(name))

    def _describe_at(self, addr):
        dims = dtype = layout = None
        for mtype, d in self._messages(addr):
            if mtype == 1:                              # dataspace
                ver, rank = d[0], d[1]
                off = 8 if ver == 1 else 4
                dims = struct.unpack_from("<" + "Q" * rank, d, off) if rank else ()
            elif mtype == 3:                            # datatype
                cls, size = d[0] & 0x0F, struct.unpack_from("<I", d, 4)[0]
                if d[0] >> 4 and cls == 1 and size in (2, 4, 8):
                    dtype = np.dtype(f"<f{size}")
                elif d[0] >> 4 and cls == 0 and size in (1, 2, 4, 8):
                    dtype = np.dtype(("<i" if d[1] & 0x08 else "<u") + str(size))
            elif mtype == 8:                            # data layout
                ver, cls = d[0], d[1]
                if ver in (3, 4) and cls == 1:
                    layout = ("contiguous",) + struct.unpack_from("<QQ", d, 2)
                elif ver in (3, 4) and cls == 0:
                    n = struct.unpack_from("<H", d, 2)[0]
                    layout = ("compact", bytes(d[4:4 + n]))
        return dims, dtype, layout

    def is_numeric(self, name):
        dims, dtype, layout = self._describe(name)
        return dims is not None and dtype is not None and layout is not None

    def read(self, name):
        """The dataset as a numpy array with the shape and element order the Julia array had (column-major data, HDF5 lists the
        dimensions slowest first, i.e. reversed)."""
        return self._read_at(self._addr(name), name)

    def _read_at(self, addr, name="<object>"):
        dims, dtype, layout = self._describe_at(addr)
        if dims is None or dtype is None or layout is None:
            raise TypeError(f"{name}: not a plain numeric dataset (Julia struct / committed datatype)")
        count = int(np.prod(dims)) if dims else 1
        if layout[0] == "contiguous":
            addr, size = layout[1], layout[2]
            if addr == UNDEF:
                return np.zeros(tuple(reversed(dims)), dtype)
            raw = np.frombuffer(self.blob, dtype, count, self.base + addr)
        else:
            raw = np.frombuffer(layout[1], dtype, count)
        return np.array(raw).reshape(tuple(reversed(dims)), order="F")


    def _object_at(self, addr):
        pos = self.base + addr
        return 0 < addr < len(self.blob) - self.base - 8 and self.blob[pos:pos + 4] == b"OHDR"

    def read_tree(self, name, _addr=None, _depth=0):
        """The numeric arrays reachable from a Julia struct stored under `name` (a `ComponentVector`'s data, the weights and biases of a
        NamedTuple of layers, ...), depth first in field order.  JLD2 stores a struct as a fixed-size record whose array-valued fields are
        8-byte references to other objects of the file; this follows every field that is such a reference without decoding the committed
        compound type, so scalars that happen to look like an object address would be followed too -- meant for parameter containers."""
        addr = self._addr(name) if _addr is None else _addr
        dims, dtype, layout = self._describe_at(addr)
        if dims is not None and dtype is not None and layout is not None:
            return [self._read_at(addr, name)]
        out = []
        if layout is not None and _depth < 8:
            raw = layout[1] if layout[0] == "compact" else self.blob[self.base + layout[1]:self.base + layout[1] + layout[2]]
            for k in range(0, len(raw) - 7, 8):
                ref = struct.unpack_from("<Q", raw, k)[0]
                if self._object_at(ref):
                    out += self.read_tree(name, ref, _depth + 1)
        return out


def load(path, *names):
    """`load(path, "X", "t")` as in FileIO / JLD2: the named plain numeric datasets (all of them without names), as a dict.
    Names may be slash paths through groups ("17/X")."""
    f = JLD2File(path)
    names = names or [k for k in f.keys() if f.is_numeric(k)]
    return {k: f.read(k) for k in names}


# ---- writer ---------------------------------------------------------------------------------------------------------------
_FLOAT_TYPE = {   # datatype message bodies JLD2 writes for Float32 / Float64 (class 1, version 3, little endian, IEEE layout)
    np.dtype("<f4"): bytes.fromhex("31201f00" "04000000" "0000" "2000" "17" "08" "00" "17" "7f000000"),
    np.dtype("<f8"): bytes.fromhex("31203f00" "08000000" "0000" "4000" "34" "0b" "00" "34" "ff030000"),
}


def _msg(mtype, body, flags=0):
    return struct.pack("<BHB", mtype, len(body), flags) + body


def _object_header(msgs):
    body = b"".join(msgs)
    w = 0 if len(body) < 256 else (1 if len(body) < 65536 else 2)
    head = b"OHDR\x02" + bytes([w]) + len(body).to_bytes(1 << w, "little") + body
    return head + struct.pack("<I", lookup3(head))


def _dataset(arr, addr):
    """Object header (+ trailing raw data for contiguous layout) of one array placed at file-relative address addr."""
    a = np.asarray(arr)
    if a.dtype not in _FLOAT_TYPE:
        raise TypeError(f"only float32 / float64 arrays can be written (got {a.dtype})")
    raw = a.tobytes(order="F")                                      # Julia's column-major element order
    dims = tuple(reversed(a.shape))                                 # HDF5 lists the slowest dimension first
    msgs = [_msg(5, b"\x03\x09"),                                   # fill value: version 3, "undefined, never written"
            _msg(1, bytes([2, len(dims), 0, 1]) + b"".join(struct.pack("<Q", n) for n in dims)),
            _msg(3, _FLOAT_TYPE[a.dtype], flags=1)]
    if len(raw) < COMPACT_BELOW:
        return _object_header(msgs + [_msg(8, b"\x04\x00" + struct.pack("<H", len(raw)) + raw)])
    probe = _object_header(msgs + [_msg(8, b"\x04\x01" + struct.pack("<QQ", 0, len(raw)))])
    head = _object_header(msgs + [_msg(8, b"\x04\x01" + struct.pack("<QQ", addr + len(probe), len(raw)))])
    return head + raw


def save(path, julia_version="1.7.3", **arrays):
    """`save(path, "X", X, "t", t, ...)` of FileIO / JLD2 for plain Float32 / Float64 arrays (keyword order = order in the file)."""
    base = 512
    text = b"HDF5-based Julia Data Format, version 0.1.1\x00 (Julia " + julia_version.encode() + b" 64-bit LE)\x00"
    out = bytearray(text.ljust(base, b"\x00"))
    body = bytearray()
    pos = 48                                                        # the superblock occupies the first 48 bytes behind the text header
    links = []
    for name, arr in arrays.items():
        obj = _dataset(arr, pos)
        links.append((name, pos))
        body += obj
        pos += len(obj)
    msgs = [_msg(2, b"\x00\x00" + b"\xff" * 16), _msg(10, b"\x00\x00")]   # link info (no dense storage), group info
    for name, addr in links:
        nb = name.encode("utf-8")
        if len(nb) > 255:
            raise ValueError("dataset names are limited to 255 bytes")
        msgs.append(_msg(6, b"\x01\x10\x01" + bytes([len(nb)]) + nb + struct.pack("<Q", addr)))
    root = _object_header(msgs)
    sb = _SIG + b"\x02\x08\x08\x00" + struct.pack("<QQQQ", base, UNDEF, base + pos + len(root), pos)
    out += sb + struct.pack("<I", lookup3(sb)) + body + root
    with open(path, "wb") as f:
        f.write(bytes(out))
