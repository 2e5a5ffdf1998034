"""Pixel-format front end (SURVEY.md 8f-4, include/itw_bcn.h section 6).

CPU: (1) the oracle restatement (oracle/itw_oracle_frontend.cpp) against the reference's OWN function bodies
(oracle/_ref/libitw_ref_frontend.so, cut from IntelPlugin.h / IntelPlugin.cpp by oracle/build_ref_frontend.py) over every
depth x plane count x format family x flag combination; (2) the kernel's per-texel routine (csrc/frontend.cuh through
tests/emu) against the oracle; (3) the restated half conversion against IEEE round-to-nearest-even where every
DirectXMath version agrees.  GPU: itw_convert_pixels / itw_encode_pixels through the C-ABI against the oracle."""
import itertools
import os

import numpy as np
import pytest

import itw_testlib as T

B = T.binding
FAMILIES = ["BC7", "BC5", "BC6H"]                     # colour / copy-plane-0 / HDR converters
SPECIALS = np.array([0.0, -0.0, 1.0, -1.0, 0.5, 1.0000001, 0.99999994, 2.0, 1e-8, 6e-8, 3e-5, 6.1e-5, 6.2e-5, 65504.0, 65519.0, 65520.0,
                     70000.0, 131000.0, 131040.0, 1e9, -5.0, np.inf, -np.inf, np.nan, 0.2, 0.21404114, 1 / 255, 254.5 / 255], np.float32)


def source(depth, planes, w, h, seed):
    rng = np.random.default_rng(seed)
    if depth == 8:
        return rng.integers(0, 256, (h, w, planes), dtype=np.uint8)
    if depth == 16:
        a = rng.integers(0, 32769, (h, w, planes), dtype=np.uint16)
        a.reshape(-1)[:8] = [0, 1, 2, 32768, 32767, 40000, 65535, 128]
        return a
    a = rng.random((h, w, planes), dtype=np.float32) * 1.2 - 0.1
    flat = a.reshape(-1)
    flat[:len(SPECIALS)] = SPECIALS[:flat.size]
    return a


def flag_sets(fmt, depth, planes):
    for alpha, gamma, fx, fy, norm in itertools.product((0, 1), (0, 1), (0, 1), (0, 1), (0, 1)):
        need = 3 if (fmt == "BC6H" and depth == 32) else 4
        if alpha and planes < need:
            continue
        if gamma and (depth != 32 or fmt == "BC6H"):
            continue
        yield alpha * 1 | gamma * 2 | fx * 4 | fy * 8 | norm * 16


def ref_convert(lib, fmt, px, flags):
    h, w, planes = px.shape
    texel = B.FORMATS[fmt][2]
    out = np.zeros((((h + 3) & ~3), ((w + 3) & ~3), 4), np.uint16 if texel == 8 else np.uint8)
    px = np.ascontiguousarray(px)
    assert lib.ref_convert_pixels(B.FORMATS[fmt][0], px.ctypes.data, w, h, planes, px.itemsize * 8, flags, out.ctypes.data) == 0
    return out


CASES = [(f, d, p) for f in FAMILIES for d in (8, 16, 32) for p in (1, 2, 3, 4)]


@pytest.mark.parametrize("fmt,depth,planes", CASES)
def test_oracle_matches_reference_function_bodies(fmt, depth, planes):
    lib = T.ref_frontend()
    o = T.oracle()
    px = source(depth, planes, 13, 7, seed=depth + planes)
    for flags in flag_sets(fmt, depth, planes):
        want = T.reference(f"convert:{fmt}:{depth}:{planes}:13x7:{flags}", lib and (lambda: ref_convert(lib, fmt, px, flags)))
        assert T.same(o.convert_pixels(fmt, px, flags), want), flags
    px = source(depth, planes, 16, 8, seed=3)                       # no padding needed
    want = T.reference(f"convert:{fmt}:{depth}:{planes}:16x8:0", lib and (lambda: ref_convert(lib, fmt, px, 0)))
    assert T.same(o.convert_pixels(fmt, px, 0), want)


@pytest.mark.parametrize("fmt,depth,planes", CASES)
def test_emulated_kernel_matches_oracle(fmt, depth, planes):
    o, e = T.oracle(), T.emu()
    px = source(depth, planes, 13, 7, seed=depth + planes)
    for flags in flag_sets(fmt, depth, planes):
        assert np.array_equal(e.convert_pixels(fmt, px, flags), o.convert_pixels(fmt, px, flags)), flags
        assert np.array_equal(e.convert_pixels(fmt, px, flags, pad=False), o.convert_pixels(fmt, px, flags, pad=False)), flags


def test_half_conversion_is_ieee_where_every_directxmath_version_agrees():
    """Results that are normal halves up to 65504: round-to-nearest-even == numpy's float16."""
    lib = T.ref_frontend()
    o = T.oracle()
    rng = np.random.default_rng(0)
    vals = np.concatenate([rng.random(4000, dtype=np.float32), (rng.random(4000, dtype=np.float32) * 65504).astype(np.float32),
                           np.float32(2.0) ** rng.integers(-14, 15, 2000).astype(np.float32) * (1 + rng.random(2000, dtype=np.float32)),
                           np.arange(256, dtype=np.float32) / np.float32(255)])
    vals = vals[(np.abs(vals) >= 6.2e-5) & (np.abs(vals) <= 65504)]
    want = vals.astype(np.float16).view(np.uint16)
    px = vals.reshape(1, -1, 1)
    got = o.convert_pixels("BC6H", px, 0, pad=False)[0, :, 0]
    assert np.array_equal(got, want)
    ref_halves = T.reference("float_to_half", lib and (lambda: np.array([lib.ref_float_to_half(float(v)) for v in vals[:2000]], np.uint16)))
    assert T.same(want[:2000], ref_halves)
    # half -> float is exact for every normal and denormal half
    hbits = np.array(list(range(0, 0x7C00, 37)) + [1, 0x3FF, 0x400, 0x7BFF], np.uint16)
    ref_floats = T.reference("half_to_float", lib and (lambda: np.array([lib.ref_half_to_float(int(b)) for b in hbits], np.float32)))
    assert T.same(hbits.view(np.float16).astype(np.float32), ref_floats)


def test_sixteen_bit_rule_is_exact_integer_arithmetic():
    """FloatToByte(v / 32768.0) == floor(v * 255 / 32768), 255 above 32768 -- all 65536 inputs."""
    o = T.oracle()
    v = np.arange(65536, dtype=np.uint16).reshape(256, 256, 1)
    got = o.convert_pixels("BC7", v, 0)[..., 0].reshape(-1)
    x = np.arange(65536, dtype=np.int64)
    want = np.where(x > 32768, 255, (x * 255) >> 15)
    assert np.array_equal(got, want)


# ---- GPU ----
@pytest.mark.gpu
@pytest.mark.parametrize("fmt,depth,planes", CASES)
def test_gpu_convert_matches_oracle(fmt, depth, planes):
    o, p = T.oracle(), T.product()
    px = source(depth, planes, 61, 35, seed=depth * 10 + planes)
    for flags in flag_sets(fmt, depth, planes):
        assert np.array_equal(p.convert_pixels(fmt, px, flags), o.convert_pixels(fmt, px, flags)), flags
    assert np.array_equal(p.convert_pixels(fmt, px, 0, pad=False), o.convert_pixels(fmt, px, 0, pad=False))
    # widths that are multiples of 4 take the four-texels-per-thread kernel; 62 -> 64 also crosses the replicated edge
    for w in (64, 62, 256):
        px = source(depth, planes, w, 10, seed=w + planes)
        for flags in list(flag_sets(fmt, depth, planes))[::3]:
            assert np.array_equal(p.convert_pixels(fmt, px, flags), o.convert_pixels(fmt, px, flags)), (w, flags)


@pytest.mark.gpu
def test_gpu_gamma_bytes_match_libm_on_a_dense_sample():
    """CUDA's double pow against glibc's through the byte conversion: 2^22 floats dense in [0, 1.05] plus every
    float next to a byte boundary (k/255)^2.2."""
    o, p = T.oracle(), T.product()
    rng = np.random.default_rng(1)
    dense = (rng.random(1 << 22, dtype=np.float32) * np.float32(1.05)).astype(np.float32)
    edges = ((np.arange(1, 256) / 255.0) ** 2.2).astype(np.float32)
    near = np.concatenate([np.nextafter(edges, np.float32(0)), edges, np.nextafter(edges, np.float32(2))])
    vals = np.concatenate([dense, near, near])[: (1 << 22) + 1024]
    vals = np.resize(vals, (2048, 2049, 1)).astype(np.float32)
    assert np.array_equal(p.convert_pixels("BC7", vals, B.FRONT_GAMMA, pad=False), o.convert_pixels("BC7", vals, B.FRONT_GAMMA, pad=False))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,prof,depth,planes,flags", [
    ("BC1", None, 8, 3, 0), ("BC3", None, 16, 4, 1), ("BC7", "alpha_veryfast", 8, 4, 1), ("BC7", "veryfast", 32, 3, 2),
    ("BC5", None, 8, 2, 4 | 8 | 16), ("BC4", None, 16, 1, 0), ("BC6H", "bc6h_veryfast", 32, 3, 0), ("BC6H", "bc6h_fast", 16, 4, 1)])
def test_gpu_encode_pixels_equals_convert_then_encode(fmt, prof, depth, planes, flags):
    """The image-level entry: same blocks as oracle-convert + oracle-encode of the padded surface."""
    o, p = T.oracle(), T.product()
    px = source(depth, planes, 50, 27, seed=11)
    if depth == 32:
        px = np.clip(np.nan_to_num(px, nan=0.5, posinf=1.0, neginf=0.0), 0, 4).astype(np.float32)
    surface = o.convert_pixels(fmt, px, flags)
    want = o.encode(fmt, surface, o.profile(prof) if prof else None)
    got = p.encode_pixels(fmt, px, flags, p.profile(prof) if prof else None)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_gpu_front_end_device_pointers_and_errors():
    import torch
    o, p = T.oracle(), T.product()
    px = source(8, 4, 128, 64, seed=2)
    want = o.convert_pixels("BC7", px, 1)
    d_src = torch.from_numpy(px.copy()).cuda()
    d_dst = torch.zeros((64, 128, 4), dtype=torch.uint8, device="cuda")
    src = B.PixelSource(d_src.data_ptr(), 128, 64, 4, 8, 0)
    p.convert_pixels_raw("BC7", src, 1, d_dst.data_ptr(), 128, 64, 128 * 4)
    assert np.array_equal(d_dst.cpu().numpy(), want)
    d_blocks = torch.zeros(32 * 16 * 16, dtype=torch.uint8, device="cuda")
    p.encode_pixels_raw("BC7", src, 1, d_blocks.data_ptr(), p.profile("alpha_veryfast"))
    assert np.array_equal(d_blocks.cpu().numpy(), o.encode("BC7", want, o.profile("alpha_veryfast")))
    with pytest.raises(RuntimeError):                       # alpha flag without an alpha plane
        p.convert_pixels("BC7", source(8, 3, 16, 16, seed=1), 1)
    with pytest.raises(RuntimeError):                       # destination of the wrong size
        p.convert_pixels_raw("BC7", src, 0, d_dst.data_ptr(), 120, 64, 128 * 4)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,dxgi,prof,depth,planes,flags,w,h,items,cube", [
    ("BC5", 83, None, 8, 3, 4 | 8 | 16, 64, 32, 1, 0),                 # normal map: flip X/Y at the top, normalise every level
    ("BC3", 77, None, 16, 4, 1, 50, 27, 1, 0),                         # odd size, alpha
    ("BC7", 98, "veryfast", 8, 3, 0, 32, 32, 6, 1),                    # cube map
    ("BC6H", 95, "bc6h_veryfast", 32, 3, 16, 32, 16, 1, 0),            # HDR normal map, wide power of two (stale-tap levels)
    ("BC6H", 95, "bc6h_veryfast", 16, 4, 1, 20, 12, 1, 0)])            # HDR, linear-filter chain
def test_gpu_whole_save_path_from_planes(fmt, dxgi, prof, depth, planes, flags, w, h, items, cube):
    """itw_dds_encode_pixels == oracle convert (+flip) -> mip chain -> oracle normalise of every level -> pad -> encode -> DDS offsets."""
    import ctypes
    import test_mips as LM
    import test_mips_f16 as HM
    o, p = T.oracle(), T.product()
    hdr = fmt == "BC6H"
    srcs = []
    for i in range(items):
        px = source(depth, planes, w, h, seed=70 + i)
        if depth == 32:
            px = np.clip(np.nan_to_num(px, nan=0.5, posinf=1.0, neginf=0.0), 0, 4).astype(np.float32)
        srcs.append(px)
    levels = LM.full_levels(w, h)
    d = B.DdsDesc(w, h, levels, items, dxgi, cube)
    s = p.profile(prof) if prof else None
    blob = p.dds_encode_pixels(d, srcs, flags, s)
    norm = flags & B.FRONT_NORMALIZE
    for item in range(items):
        top = o.convert_pixels(fmt, srcs[item], flags & ~B.FRONT_NORMALIZE, pad=False)
        srgb = 1 if dxgi in (72, 78, 99) else 0                    # *_SRGB encodings take the sRGB-correct chain (IntelPlugin.cpp:152-154)
        chain = HM.oracle_chain(top, levels) if hdr else T.oracle_mip_chain_rgba8(top, srgb, levels, pad=False)
        for mip in range(levels):
            lv = np.ascontiguousarray(chain[mip])
            if norm:                                               # the oracle's normalise pass through an identity conversion
                if hdr:
                    rgb = o.convert_pixels(fmt, lv.view(np.float16).astype(np.float32), B.FRONT_NORMALIZE, pad=False)
                    lv = np.concatenate([rgb[..., :3], lv[..., 3:]], axis=2)
                else:
                    lv = o.convert_pixels(fmt, lv, B.FRONT_NORMALIZE | B.FRONT_HAS_ALPHA, pad=False)
            padded = HM.pad4(lv)
            want = o.encode(fmt, np.ascontiguousarray(padded), o.profile(prof) if prof else None)
            off = p.lib.itw_dds_image_offset(ctypes.byref(d), item, mip)
            assert np.array_equal(blob[off:off + want.size], want), (item, mip)


def test_oracle_matches_committed_reference_digests():
    """The digests were produced by the reference's own function bodies (tests/golden/make_golden_frontend.py); they keep the
    oracle pinned where neither /root/reference nor a prebuilt oracle/_ref exists."""
    import hashlib
    import json
    import os
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "frontend_digests.json")))
    o = T.oracle()
    n = 0
    for fmt, depth, planes in CASES:
        px = source(depth, planes, 13, 7, seed=depth + planes)
        for flags in flag_sets(fmt, depth, planes):
            got = hashlib.sha256(o.convert_pixels(fmt, px, flags).tobytes()).hexdigest()
            assert got == golden["convert"][f"{fmt}:{depth}:{planes}:{flags}"], (fmt, depth, planes, flags)
            n += 1
    assert n == len(golden["convert"])


def test_gamma_table_equals_pow_around_every_threshold_and_on_a_dense_sample():
    """The kernel evaluates the 32-bit gamma conversion from a threshold table (csrc/gamma_table.cuh) instead of pow: the
    emulated routine must equal the oracle (C library pow) on both float neighbours of all 255 thresholds, on a dense
    sample of [0, 1.05] and on the special values."""
    import re
    o, e = T.oracle(), T.emu()
    text = open(os.path.join(T.ROOT, "intel-texture-works-plugin_b200", "csrc", "gamma_table.cuh")).read()
    bits = np.array([int(x, 16) for x in re.findall(r"0x([0-9A-F]{8})u", text)], np.uint32)
    assert bits.size == 255 and np.all(np.diff(bits.astype(np.int64)) > 0)
    near = np.concatenate([bits - 2, bits - 1, bits, bits + 1, bits + 2]).view(np.float32)
    rng = np.random.default_rng(5)
    dense = (rng.random(1 << 20, dtype=np.float32) * np.float32(1.05)).astype(np.float32)
    tiny = (rng.random(4096, dtype=np.float32) * np.float32(1e-4)).astype(np.float32)
    vals = np.concatenate([near, dense, tiny, SPECIALS, -SPECIALS])
    vals = np.resize(vals, (1027, 1024, 1)).astype(np.float32)
    got = e.convert_pixels("BC7", vals, B.FRONT_GAMMA, pad=False)
    want = o.convert_pixels("BC7", vals, B.FRONT_GAMMA, pad=False)
    assert np.array_equal(got, want)
