"""BC6H / BC7 decoders pinned to the reference's own code (SURVEY.md 8f-3).

oracle/build_ref_decode.py cuts D3DX_BC6H::Decode / D3DX_BC7::Decode (DirectXTex/BC6HBC7.cpp:1077-1236, :1937-2144) and
their tables out of /root/reference and compiles them behind a shim.  Against those bodies, block by block:
  * tests/bcn_decode.py -- the independent numpy decoders every other decode test leans on,
  * csrc/decode.cuh run on the CPU (tests/emu) -- UF16, SF16 (D3DXDecodeBC6HS) and BC7,
  * (-m gpu) the decode kernels through itw_decode.
Inputs: encoder output of every profile (every mode the encoders emit) and random bit patterns under every mode field,
the reserved ones included.  DirectXTex returns floats: BC7 texels are byte * (1/255) -- the test checks that the byte the
product returns maps to exactly that float; BC6H texels are XMConvertHalfToFloat of the half bits the product returns."""
import ctypes
import os
import sys

import numpy as np
import pytest

import bcn_decode as D
import itw_testlib as T
from test_decode import LAYOUTS, random_blocks, reference_decode


def dx():
    """DirectXTex's own BC6H / BC7 decoders, or None where they are not built."""
    sys.path.insert(0, os.path.join(T.ROOT, "oracle"))
    try:
        import build_ref_decode
        try:
            path = build_ref_decode.build(verbose=False)
        except FileNotFoundError:
            return None
    finally:
        sys.path.pop(0)
    lib = ctypes.CDLL(path)
    lib.ref_decode_blocks.restype = None
    lib.ref_decode_blocks.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
    return lib


def dx_decode(lib, fmt_id, blocks, tag):
    """D3DX_BC6H / D3DX_BC7 Decode of every block: (n, 16, 4) floats, or their stored digest where `lib` is None."""
    def decode():
        b = np.ascontiguousarray(np.frombuffer(bytes(blocks), np.uint8))
        n = b.size // 16
        out = np.zeros((n, 16, 4), np.float32)
        lib.ref_decode_blocks(fmt_id, b.ctypes.data, n, out.ctypes.data)
        return out
    return T.reference(f"dx_decode:{fmt_id}:{tag}", lib and decode)


def as_blocks(img, w, h):
    """H x W x 4 image -> (n blocks, 16 texels, 4) in raster block order"""
    return img.reshape(h // 4, 4, w // 4, 4, 4).transpose(0, 2, 1, 3, 4).reshape(-1, 16, 4)


def check_bc7(got_bytes, want_floats, tag):
    g = got_bytes.astype(np.float32) * np.float32(1.0 / 255.0)            # HDRColorA(const LDRColorA&), BC.h:151-157
    assert T.same(g, want_floats), f"{tag}: differs from D3DXDecodeBC7" + _first_blocks(g, want_floats)


def half_bits_to_float(bits):
    """XMConvertHalfToFloat of DirectXMath 3.06 (the reference's SDK): IEEE for every finite half; exponent 31 is an ORDINARY
    binade there (0xFC00 -> -65536, not -inf).  A signed 16-bit-endpoint block can reach it: -32768 un-quantises to -0x7C00."""
    b = bits.astype(np.uint16)
    f = b.view(np.float16).astype(np.float32)
    top = (b & 0x7C00) == 0x7C00
    mag = (np.float32(1.0) + (b & 0x3FF).astype(np.float32) / np.float32(1024.0)) * np.float32(65536.0)
    return np.where(top, np.where(b & 0x8000, -mag, mag), f).astype(np.float32)


def check_bc6(got_half_bits, want_floats, tag):
    g = half_bits_to_float(got_half_bits)
    assert T.same(g, want_floats), f"{tag}: differs from D3DXDecodeBC6H" + _first_blocks(g, want_floats)


def _first_blocks(g, want_floats):
    if isinstance(want_floats, str):
        return " (stored digest)"
    bad = np.nonzero((g != want_floats).any(axis=(1, 2)))[0]
    return f": {bad.size} blocks, first {bad[:5]}"


def streams(fmt):
    """(tag, blocks, width, height): encoder output of EVERY profile on three corpus images + random bits (every mode field)"""
    o = T.oracle()
    corpus = T.corpus_for(fmt)
    profs = T.binding.BC7_PROFILES if fmt == "BC7" else T.binding.BC6H_PROFILES
    names = ("gradient", "smooth", "random", "alpha01", "twocolour") if fmt == "BC7" else ("smooth", "lowvar", "random", "narrow", "signbits")
    for prof in profs:
        for name in names:
            yield f"{prof}-{name}", T.run(o, fmt, corpus[name], prof), 64, 64
    yield "random-bits", random_blocks(fmt, 64 * 72, seed=21), 256, 288
    rng = np.random.default_rng(4)
    ext = rng.integers(0, 256, (64 * 16, 16), dtype=np.uint8)
    ext[:, 1:11] = np.where(rng.random((64 * 16, 10)) < 0.5, 0xFF, 0x00).astype(np.uint8)     # saturated / zero endpoint fields
    for i in range(ext.shape[0]):
        ext[i, 0] = (ext[i, 0] & 0xE0) | (i % 32) if fmt == "BC6H" else ext[i, 0]
    yield "extreme-endpoints", ext.reshape(-1), 256, 64


def test_numpy_decoders_equal_directxtex():
    """tests/bcn_decode.py (BC7, BC6H unsigned) is what test_decode.py, smoke() and the PSNR gates trust: pin it."""
    lib = dx()
    for fmt, fid, check in (("BC7", 98, check_bc7), ("BC6H", 95, check_bc6)):
        for tag, blocks, w, h in streams(fmt):
            if w * h > 64 * 64:
                blocks, w, h = blocks[: 16 * 16 * 16], 64, 64               # the numpy decoders are slow: 256 blocks of the big sets
                tag += ":first256"
            got = reference_decode(fmt, blocks, w, h)
            check(as_blocks(got, w, h), dx_decode(lib, fid, blocks, tag), f"{fmt} {tag}")


@pytest.mark.parametrize("fmt,fid", [("BC7", 98), ("BC6H", 95), ("BC6H_SF16", 96)])
def test_kernel_decode_logic_equals_directxtex(fmt, fid):
    """csrc/decode.cuh on the CPU (tests/emu), every block of every stream; SF16 = D3DXDecodeBC6HS on the same bit patterns."""
    lib, e = dx(), T.emu()
    base = "BC6H" if fmt.startswith("BC6H") else fmt
    for tag, blocks, w, h in streams(base):
        got = emu_decode(e, fid, blocks, w, h)
        (check_bc7 if base == "BC7" else check_bc6)(as_blocks(got, w, h), dx_decode(lib, fid, blocks, tag), f"{fmt} {tag}")


def emu_decode(api, fid, blocks, w, h):
    blocks = np.ascontiguousarray(np.frombuffer(bytes(blocks), np.uint8))
    img = np.zeros((h, w, 4), np.uint16 if fid in (95, 96) else np.uint8)
    f = api.fn("itw_decode")
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.POINTER(T.binding.RgbaSurface)]
    surf = T.binding.RgbaSurface(img.ctypes.data, w, h, img.strides[0])
    assert f(fid, blocks.ctypes.data, ctypes.byref(surf)) == 0
    return img


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,fid", [("BC7", 98), ("BC6H", 95), ("BC6H_SF16", 96)])
def test_gpu_decode_equals_directxtex(fmt, fid):
    lib, p = dx(), T.product()
    base = "BC6H" if fmt.startswith("BC6H") else fmt
    for tag, blocks, w, h in list(streams(base)) + [("random-bits-large", random_blocks(base, 256 * 256, seed=77), 1024, 1024)]:
        got = emu_decode(p, fid, blocks, w, h)
        p.check()
        (check_bc7 if base == "BC7" else check_bc6)(as_blocks(got, w, h), dx_decode(lib, fid, blocks, tag), f"{fmt} {tag}")
