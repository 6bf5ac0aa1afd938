"""PCD reader / writer of the facade (pcl_b200/pcl_compat/pcl/io/pcd_io.h): CPU-only.

* the C++ self-test (LZF coder, ascii / binary / binary_compressed round trips, organised clouds, foreign field types);
* the reference's own fixtures (tests/golden/pcd/, written by tests/golden/make_pcd_fixtures.py: the large ones cut to
  their first points and compressed again by the reference's LZF coder), decoded here by an independent pure-Python
  LZF + plane unpacking and compared bit for bit with what the C++ reader returns;
* the ASCII fixtures against the committed golden vectors."""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, "pcl_b200", "pcl_compat")
EXE = os.path.join(COMPAT, "tests", "test_pcd_io")
REF = os.path.join(ROOT, "tests", "golden", "pcd")


@pytest.fixture(scope="module")
def exe():
    subprocess.check_call(["make", "-C", COMPAT, "-s", "tests/test_pcd_io"])
    return EXE


def _dump(exe, path, tmp):
    out = os.path.join(tmp, "dump.bin")
    subprocess.check_call([exe, "dump", path, out])
    raw = open(out, "rb").read()
    n, w, h, dense = struct.unpack("<QIII", raw[:20])
    return np.frombuffer(raw[20:], dtype=np.float32).reshape(n, 3), w, h, bool(dense)


def _lzf_decompress(data, out_len):
    """LZF stream format: ctrl < 32 -> ctrl + 1 literals; else length (ctrl >> 5) + 2 (7 -> + next byte) at distance
    ((ctrl & 31) << 8 | next) + 1."""
    out = bytearray()
    i, n = 0, len(data)
    while i < n:
        ctrl = data[i]
        i += 1
        if ctrl < 32:
            out += data[i:i + ctrl + 1]
            i += ctrl + 1
        else:
            length = ctrl >> 5
            if length == 7:
                length += data[i]
                i += 1
            dist = ((ctrl & 0x1f) << 8 | data[i]) + 1
            i += 1
            length += 2
            start = len(out) - dist
            assert start >= 0
            if dist >= length:
                out += out[start:start + length]
            else:
                for k in range(length):
                    out.append(out[start + k])
    assert len(out) == out_len
    return bytes(out)


def _read_pcd_python(path):
    raw = open(path, "rb").read()
    pos, hdr = 0, {}
    while True:
        end = raw.index(b"\n", pos)
        line = raw[pos:end].decode("ascii", "replace").strip()
        pos = end + 1
        if not line or line.startswith("#"):
            continue
        key, *vals = line.split()
        hdr[key] = vals
        if key == "DATA":
            break
    names = hdr.get("FIELDS", hdr.get("COLUMNS"))
    sizes = [int(v) for v in hdr.get("SIZE", ["4"] * len(names))]
    types = hdr.get("TYPE", ["F"] * len(names))
    counts = [int(v) for v in hdr.get("COUNT", ["1"] * len(names))]
    npts = int(hdr["POINTS"][0])
    mode = hdr["DATA"][0]
    cols = {}
    if mode == "binary_compressed":
        csize, usize = struct.unpack("<II", raw[pos:pos + 8])
        buf = _lzf_decompress(raw[pos + 8:pos + 8 + csize], usize)
        off = 0
        for nm, sz, ty, ct in zip(names, sizes, types, counts):
            if nm == "_":
                continue
            if ty == "F" and sz == 4:
                cols[nm] = np.frombuffer(buf, dtype=np.float32, count=npts * ct, offset=off).reshape(npts, ct)[:, 0]
            off += sz * ct * npts
    elif mode == "binary":
        step = sum(s * c for s, c in zip(sizes, counts))
        rec = np.frombuffer(raw, dtype=np.uint8, count=npts * step, offset=pos).reshape(npts, step)
        off = 0
        for nm, sz, ty, ct in zip(names, sizes, types, counts):
            if ty == "F" and sz == 4 and nm != "_":
                cols[nm] = rec[:, off:off + 4].copy().view(np.float32)[:, 0]
            off += sz * ct
    else:
        body = np.array([[float(t) for t in ln.split()] for ln in raw[pos:].decode().splitlines() if ln.strip()], dtype=np.float64)
        col = 0
        for nm, ct in zip(names, counts):
            cols[nm] = body[:, col].astype(np.float32)
            col += ct
    w = int(hdr["WIDTH"][0]) if "WIDTH" in hdr else npts
    h = int(hdr["HEIGHT"][0]) if "HEIGHT" in hdr else 1
    return np.stack([cols["x"], cols["y"], cols["z"]], 1), w, h


def test_cpp_selftest(exe, tmp_path):
    r = subprocess.run([exe, "selftest", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "PASSED" in r.stdout


@pytest.mark.parametrize("name", ["milk.pcd", "cturtle.pcd", "car6.pcd", "noisy_slice_displaced.pcd", "colored_cloud.pcd",
                                  "office1_keypoints.pcd", "bun0.pcd", "bun4.pcd", "sac_plane_test.pcd"])
def test_reference_fixtures_decode_identically(exe, tmp_path, name):
    path = os.path.join(REF, name)
    want, w, h = _read_pcd_python(path)
    got, gw, gh, dense = _dump(exe, path, str(tmp_path))
    assert (gw, gh) == (w, h) and got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))  # bit for bit, NaNs included
    assert dense == bool(np.isfinite(want).all()) or not dense  # other fields of the file may hold the NaNs
    # our three writers reproduce the cloud
    for mode in ("ascii", "binary", "compressed"):
        out = os.path.join(str(tmp_path), "re.pcd")
        subprocess.check_call([exe, "recode", path, out, mode])
        again, aw, ah, _ = _dump(exe, out, str(tmp_path))
        assert (aw, ah) == (w, h)
        assert np.array_equal(again.view(np.uint32), want.view(np.uint32)) or (
            mode == "ascii" and np.array_equal(np.isnan(again), np.isnan(want)) and np.allclose(again, want, rtol=0, atol=0, equal_nan=True))
        # and the Python reader agrees on what our writers put on disk (writer <-> independent reader)
        py, pw, ph = _read_pcd_python(out)
        assert (pw, ph) == (w, h) and np.array_equal(np.isnan(py), np.isnan(want))
        assert np.array_equal(py[~np.isnan(py)], want[~np.isnan(want)])


@pytest.mark.parametrize("name", ["milk.pcd", "cturtle.pcd", "car6.pcd", "noisy_slice_displaced.pcd", "colored_cloud.pcd",
                                  "office1_keypoints.pcd", "bun0.pcd", "sac_plane_test.pcd"])
def test_reference_fixtures_through_the_blob_reader(exe, tmp_path, name):
    """PCDReader::read into a pcl::PCLPointCloud2 + fromPCLPointCloud2 (the route tools/iterative_closest_point.cpp takes):
    the same coordinates as the independent Python decoder, bit for bit."""
    path = os.path.join(REF, name)
    want, w, h = _read_pcd_python(path)
    out = os.path.join(str(tmp_path), "blob.bin")
    subprocess.check_call([exe, "dumpblob", path, out])
    raw = open(out, "rb").read()
    n, gw, gh, dense = struct.unpack("<QIII", raw[:20])
    got = np.frombuffer(raw[20:], dtype=np.float32).reshape(n, 3)
    assert (gw, gh) == (w, h) and got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert not dense or bool(np.isfinite(want).all())


@pytest.mark.parametrize("header,body", [
    ("FIELDS a x y\nSIZE -4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 2\nHEIGHT 1\nPOINTS 2\nDATA binary\n", b"\0" * 32),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 4000000000\nHEIGHT 1\nPOINTS 4000000000\nDATA binary\n", b"\0" * 12),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 100\nHEIGHT 1\nPOINTS 100\nDATA binary_compressed\n",
     struct.pack("<II", 4, 4000000000) + b"\0" * 4),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 100\nHEIGHT 1\nPOINTS 100\nDATA binary_compressed\n",
     struct.pack("<II", 4, 1200) + b"\0" * 4),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 4000000000\nHEIGHT 1\nPOINTS 4000000000\nDATA binary_compressed\n",
     struct.pack("<II", 4, 4000000000) + b"\0" * 4),
])
def test_malformed_files_are_rejected_by_the_blob_reader(exe, tmp_path, header, body):
    f = tmp_path / "bad.pcd"
    f.write_bytes(header.encode() + body)
    r = subprocess.run([exe, "dumpblob", str(f), str(tmp_path / "o.bin")], capture_output=True, text=True)
    assert r.returncode == 2, (r.returncode, r.stderr)


def test_ascii_fixtures_match_golden(exe, tmp_path, golden):
    for name, key in (("bun0.pcd", "bun0"), ("bun4.pcd", "bun4"), ("sac_plane_test.pcd", "sac_plane")):
        got, w, h, dense = _dump(exe, os.path.join(REF, name), str(tmp_path))
        assert h == 1 and w == got.shape[0]
        assert dense == (name != "sac_plane_test.pcd")  # that file carries NaN normals: every field counts (pcd_io.cpp:636-665)
        assert np.array_equal(got, golden[key][:w, :3].astype(np.float32))  # the stored sac_plane_test.pcd is its first 400 points


@pytest.mark.parametrize("header,body", [
    # negative SIZE: used to wrap a field offset to 2^64-4 and read outside the buffer
    ("FIELDS a x y\nSIZE -4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 2\nHEIGHT 1\nPOINTS 2\nDATA binary\n", b"\0" * 32),
    ("FIELDS x y z\nSIZE 4 4 3\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 1\nHEIGHT 1\nPOINTS 1\nDATA binary\n", b"\0" * 16),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 0 1\nWIDTH 1\nHEIGHT 1\nPOINTS 1\nDATA binary\n", b"\0" * 16),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F Q\nCOUNT 1 1 1\nWIDTH 1\nHEIGHT 1\nPOINTS 1\nDATA binary\n", b"\0" * 16),
    # a tiny file that asks for a huge allocation
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 4000000000\nHEIGHT 1\nPOINTS 4000000000\nDATA binary\n", b"\0" * 12),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 4000000000\nHEIGHT 1\nPOINTS 4000000000\nDATA ascii\n", b"1 2 3\n"),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 100\nHEIGHT 1\nPOINTS 100\nDATA binary_compressed\n",
     struct.pack("<II", 4, 4000000000) + b"\0" * 4),
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 18446744073709551615\nHEIGHT 3\nPOINTS 5\nDATA ascii\n", b""),
    # compressed body of 12 bytes that claims four billion points: refused before any allocation
    ("FIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 4000000000\nHEIGHT 1\nPOINTS 4000000000\nDATA binary_compressed\n",
     struct.pack("<II", 4, 4000000000) + b"\0" * 4),
])
def test_malformed_headers_are_rejected(exe, tmp_path, header, body):
    """Untrusted files: bad SIZE / COUNT / TYPE and point counts the file cannot hold are refused (exit code 2 of the
    dump tool = loadPCDFile returned -1) instead of wrapping offsets, reading out of bounds or allocating gigabytes."""
    f = tmp_path / "bad.pcd"
    f.write_bytes(("# .PCD v0.7\nVERSION 0.7\n" + header).encode() + body)
    r = subprocess.run([exe, "dump", str(f), str(tmp_path / "o.bin")], capture_output=True, timeout=20)
    assert r.returncode == 2, (r.returncode, r.stderr[-300:])
