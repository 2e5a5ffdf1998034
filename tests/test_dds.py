"""DDS container (SURVEY.md 8f-1).  The expected header bytes are derived by hand from the layout in
DirectXTex/DDS.h:40-235 and the rules of _EncodeDDSHeader (DirectXTexDDS.cpp:441-675); the parser below is
independent of the library's own reader."""
import ctypes
import struct

import numpy as np
import pytest

import itw_testlib as T

D = T.binding.DdsDesc


def parse(blob):
    magic, size, flags, height, width, pitch, depth, mips = struct.unpack_from("<8I", blob, 0)
    pf_size, pf_flags, fourcc = struct.unpack_from("<3I", blob, 4 + 72)
    caps, caps2 = struct.unpack_from("<2I", blob, 4 + 104)
    out = dict(magic=magic, size=size, flags=flags, height=height, width=width, pitch=pitch, depth=depth, mips=mips,
               pf_size=pf_size, pf_flags=pf_flags, fourcc=struct.pack("<I", fourcc), caps=caps, caps2=caps2)
    if out["fourcc"] == b"DX10":
        out["dx10"] = struct.unpack_from("<5I", blob, 128)
    return out


def header(lib, desc):
    n = lib.lib.itw_dds_header_bytes(ctypes.byref(desc))
    buf = np.zeros(n, np.uint8)
    assert lib.lib.itw_dds_write_header(ctypes.byref(desc), buf.ctypes.data, n) == n
    return buf.tobytes()


def test_legacy_header_bc1_single_level():
    lib = T.product()
    h = header(lib, D(256, 256, 1, 1, 71, 0))
    assert len(h) == 128
    p = parse(h)
    assert p == dict(magic=0x20534444, size=124, flags=0x1007 | 0x20000 | 0x80000, height=256, width=256, pitch=64 * 64 * 8,
                     depth=1, mips=1, pf_size=32, pf_flags=4, fourcc=b"DXT1", caps=0x1000, caps2=0)
    assert h[4 + 28:4 + 72] == bytes(44)                       # dwReserved1[11]
    assert h[4 + 112:] == bytes(12)                            # caps3, caps4, reserved2


def test_dx10_header_bc7_srgb_full_mip_chain():
    lib = T.product()
    d = D(512, 256, 10, 1, 99, 0)
    h = header(lib, d)
    assert len(h) == 148
    p = parse(h)
    assert (p["fourcc"], p["mips"], p["caps"], p["pitch"]) == (b"DX10", 10, 0x1000 | 0x400008, 128 * 64 * 16)
    assert p["dx10"] == (99, 3, 0, 1, 0)
    # payload: levels 512x256 ... 1x1, blocks = ceil(w/4)*ceil(h/4)
    sizes = [((max(512 >> l, 1) + 3) // 4) * ((max(256 >> l, 1) + 3) // 4) * 16 for l in range(10)]
    assert [lib.lib.itw_dds_image_bytes(ctypes.byref(d), l) for l in range(10)] == sizes
    assert [lib.lib.itw_dds_image_offset(ctypes.byref(d), 0, l) for l in range(10)] == [148 + sum(sizes[:l]) for l in range(10)]
    assert lib.lib.itw_dds_file_bytes(ctypes.byref(d)) == 148 + sum(sizes)


def test_cubemap_and_format_table():
    lib = T.product()
    d = D(64, 64, 7, 6, 77, 1)
    p = parse(header(lib, d))
    assert (p["fourcc"], p["caps"], p["caps2"]) == (b"DXT5", 0x1000 | 0x400008 | 0x8, 0xFE00)
    per_face = sum(((max(64 >> l, 1) + 3) // 4) ** 2 * 16 for l in range(7))
    assert lib.lib.itw_dds_image_offset(ctypes.byref(d), 3, 2) == 128 + 3 * per_face + (16 * 16 + 8 * 8) * 16
    # which formats get the legacy FourCC and which the DX10 extension (DirectXTexDDS.cpp:479-486)
    want = {71: b"DXT1", 72: b"DX10", 77: b"DXT5", 78: b"DX10", 80: b"BC4U", 83: b"BC5U", 95: b"DX10", 96: b"DX10", 98: b"DX10", 99: b"DX10"}
    for fmt, cc in want.items():
        assert parse(header(lib, D(16, 16, 1, 1, fmt, 0)))["fourcc"] == cc, fmt
    # a 2-element array is not expressible in the legacy header
    assert parse(header(lib, D(16, 16, 1, 2, 71, 0)))["fourcc"] == b"DX10"
    # unsupported descriptions are refused
    for bad in (D(16, 16, 1, 1, 28, 0), D(16, 16, 6, 1, 71, 0), D(0, 16, 1, 1, 71, 0), D(16, 16, 1, 5, 71, 1)):
        assert lib.lib.itw_dds_header_bytes(ctypes.byref(bad)) == 0


def test_reader_round_trip():
    lib = T.product()
    for d in (D(256, 256, 1, 1, 71, 0), D(512, 256, 10, 1, 99, 0), D(64, 64, 7, 6, 77, 1), D(32, 32, 1, 12, 98, 1), D(8, 8, 1, 3, 95, 0)):
        h = np.frombuffer(header(lib, d), np.uint8).copy()
        back = D()
        off = lib.lib.itw_dds_read_header(h.ctypes.data, h.size, ctypes.byref(back))
        assert off == h.size
        assert [getattr(back, f) for f, _ in D._fields_] == [getattr(d, f) for f, _ in D._fields_]
    junk = np.zeros(148, np.uint8)
    assert lib.lib.itw_dds_read_header(junk.ctypes.data, 148, ctypes.byref(D())) == 0


@pytest.mark.gpu
def test_encode_file_equals_per_level_encodes():
    """The whole save path for one texture: BC3 cube map with mips and BC7 sRGB 2-D texture, every level
    encoded straight into the blob; payload must equal the per-level CompressBlocks* output."""
    lib = T.product()
    faces = [T.synth.mip_chain(T.synth.mixed_rgba8(64, 64, seed=s)) for s in range(6)]
    d = D(64, 64, 7, 6, 77, 1)
    blob = lib.dds_encode_file(d, [lvl for f in faces for lvl in f])
    assert parse(blob.tobytes())["fourcc"] == b"DXT5"
    for item in range(6):
        for mip in range(7):
            off = lib.lib.itw_dds_image_offset(ctypes.byref(d), item, mip)
            want = lib.encode("BC3", np.ascontiguousarray(faces[item][mip]))
            assert np.array_equal(blob[off:off + want.size], want), (item, mip)
    chain = T.synth.mip_chain(T.synth.random_rgba8(64, 128, seed=9))    # 128 wide, 64 high
    d = D(128, 64, 8, 1, 99, 0)
    s = lib.profile("veryfast")
    blob = lib.dds_encode_file(d, chain, s)
    for mip in range(8):
        off = lib.lib.itw_dds_image_offset(ctypes.byref(d), 0, mip)
        want = lib.encode("BC7", np.ascontiguousarray(chain[mip]), s)
        assert np.array_equal(blob[off:off + want.size], want), mip


def test_header_equals_directxtex_header_encoder():
    """itw_dds_write_header against the reference's OWN _EncodeDDSHeader body (DirectXTexDDS.cpp:441-675 + DDS.h, cut by
    oracle/build_ref_dds.py): every block-compressed format the library writes x sizes x mip counts x plain / cube / array."""
    import ctypes
    import os
    import sys
    sys.path.insert(0, os.path.join(T.ROOT, "oracle"))
    try:
        import build_ref_dds
        try:
            ref = ctypes.CDLL(build_ref_dds.build(verbose=False))
            ref.ref_dds_header.restype = ctypes.c_size_t
            ref.ref_dds_header.argtypes = [ctypes.c_uint32] * 6 + [ctypes.c_void_p, ctypes.c_size_t]
        except FileNotFoundError:                                  # not built here: its stored digest stands in
            ref = None
    finally:
        sys.path.pop(0)
    lib = T.product().lib
    cases = [(fmt, w, h, mips, items, cube)
             for fmt in (71, 72, 77, 78, 80, 83, 95, 96, 98, 99)
             for (w, h) in ((256, 256), (60, 36), (1, 1), (4096, 2048), (5, 300))
             for mips in (1, 2, 5) if mips <= max(w, h).bit_length()          # no more levels than the size has
             for (items, cube) in ((1, 0), (6, 1), (3, 0), (12, 1))]
    assert len(cases) == 520

    def headers(write):
        """(n, 160) header bytes, zero beyond each header's size; the size is the first two bytes' little-endian value"""
        out = np.zeros((len(cases), 162), np.uint8)
        for row, c in zip(out, cases):
            size = write(c, row[2:])
            assert size in (128, 148), c
            row[:2] = (size & 255, size >> 8)
            row[2 + size:] = 0
        return out

    def ours(c, buf):
        d = D(c[1], c[2], c[3], c[4], c[0], c[5])
        size = lib.itw_dds_header_bytes(ctypes.byref(d))
        assert lib.itw_dds_write_header(ctypes.byref(d), buf.ctypes.data, 160) == size, c
        return size
    got = headers(ours)
    want = T.reference("dds_header:520_cases", ref and (lambda: headers(
        lambda c, buf: ref.ref_dds_header(c[1], c[2], c[3], c[4], c[0], c[5], buf.ctypes.data, 160))))
    assert T.same(got, want), "" if isinstance(want, str) else [cases[i] for i in np.nonzero((got != want).any(1))[0][:5]]


def test_reader_survives_corrupted_and_random_headers():
    """itw_dds_read_header parses untrusted bytes: mutated valid headers and random buffers, truncated at random, must be
    rejected or yield a description the library can size -- never crash."""
    import ctypes
    lib = T.product().lib
    d = D(64, 64, 3, 1, 98, 0)
    n = lib.itw_dds_header_bytes(ctypes.byref(d))
    good = np.zeros(200, np.uint8)
    lib.itw_dds_write_header(ctypes.byref(d), good.ctypes.data, 200)
    rng = np.random.default_rng(0)
    out = D()
    accepted = 0
    for _ in range(20000):
        b = good.copy()
        for _ in range(int(rng.integers(1, 6))):
            b[rng.integers(0, n)] = rng.integers(0, 256)
        if lib.itw_dds_read_header(b.ctypes.data, int(rng.integers(0, n + 8)), ctypes.byref(out)):
            accepted += 1
            assert lib.itw_dds_file_bytes(ctypes.byref(out)) > 0
    assert accepted > 0
    for _ in range(20000):
        b = rng.integers(0, 256, 200, dtype=np.uint8)
        b[:4] = good[:4]
        lib.itw_dds_read_header(b.ctypes.data, int(rng.integers(0, 200)), ctypes.byref(out))
