#!/usr/bin/env python3
"""Regenerates tests/golden/pcd/ from a PCL checkout's own test/*.pcd files (the fixtures of tests/test_pcd_io.py).

    make -C oracle ref PCL_SRC=<PCL checkout>      # the reference's LZF coder, io/src/lzf.cpp
    python tests/golden/make_pcd_fixtures.py <PCL checkout>

The files of VERBATIM are copied byte for byte.  Those of SAMPLE_POINTS, too large to store whole, keep their header
and their first SAMPLE_POINTS[name] points: an ASCII file keeps its first data lines, a binary_compressed file is decompressed and its planes
cut and compressed again by PCL's own lzfCompress, laid out as PCDWriter::writeBinaryCompressed lays it out
(pcd_io.cpp: uint32 compressed size, uint32 raw size, LZF stream of the field planes)."""
import ctypes as C
import os
import shutil
import struct
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(ROOT, "tests", "golden", "pcd")
VERBATIM = ["noisy_slice_displaced.pcd", "colored_cloud.pcd", "office1_keypoints.pcd", "bun0.pcd", "bun4.pcd"]
SAMPLE_POINTS = {"milk.pcd": 3000, "car6.pcd": 3000, "cturtle.pcd": 3000, "sac_plane_test.pcd": 400}


def _header(raw):
    """(header lines, offset of the body, {key: values})."""
    pos, lines, hdr = 0, [], {}
    while True:
        end = raw.index(b"\n", pos)
        line = raw[pos:end]
        lines.append(line)
        pos = end + 1
        s = line.decode("ascii").strip()
        if s and not s.startswith("#"):
            key, *vals = s.split()
            hdr[key] = vals
            if key == "DATA":
                return lines, pos, hdr


def _with_count(lines, n):
    out = []
    for ln in lines:
        key = ln.split(b" ", 1)[0]
        out.append(key + b" %d" % n if key in (b"WIDTH", b"POINTS") else ln)
    return b"\n".join(out) + b"\n"


def sample(lzf, raw, n):
    lines, pos, hdr = _header(raw)
    assert hdr.get("HEIGHT", ["1"]) == ["1"]
    total = int(hdr["POINTS"][0])
    if hdr["DATA"][0] == "ascii":
        rows = raw[pos:].split(b"\n")[:n]
        return _with_count(lines, n) + b"\n".join(rows) + b"\n"
    assert hdr["DATA"][0] == "binary_compressed"
    csize, usize = struct.unpack("<II", raw[pos:pos + 8])
    buf = C.create_string_buffer(usize)
    assert lzf._ZN3pcl13lzfDecompressEPKvjPvj(raw[pos + 8:pos + 8 + csize], csize, buf, usize) == usize
    widths = [int(s) * int(c) for s, c in zip(hdr["SIZE"], hdr["COUNT"])]
    planes, off = [], 0
    for w in widths:
        planes.append(buf.raw[off:off + w * n])
        off += w * total
    data = b"".join(planes)
    out = C.create_string_buffer(len(data) * 3 // 2)
    m = lzf._ZN3pcl11lzfCompressEPKvjPvj(data, len(data), out, len(out))
    assert m > 0
    return _with_count(lines, n) + struct.pack("<II", m, len(data)) + out.raw[:m]


def main():
    test = os.path.join(sys.argv[1], "test")
    lzf = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "liblzf.so"))
    for f in (lzf._ZN3pcl11lzfCompressEPKvjPvj, lzf._ZN3pcl13lzfDecompressEPKvjPvj):
        f.restype = C.c_uint
        f.argtypes = [C.c_char_p, C.c_uint, C.c_void_p, C.c_uint]
    os.makedirs(OUT, exist_ok=True)
    for name in VERBATIM:
        shutil.copyfile(os.path.join(test, name), os.path.join(OUT, name))
    for name, n in SAMPLE_POINTS.items():
        with open(os.path.join(test, name), "rb") as f:
            data = sample(lzf, f.read(), n)
        with open(os.path.join(OUT, name), "wb") as f:
            f.write(data)
    for name in sorted(os.listdir(OUT)):
        print(name, os.path.getsize(os.path.join(OUT, name)))


if __name__ == "__main__":
    main()
