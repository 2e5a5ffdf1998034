"""The on-GPU pre-pass -- mip chain plus pad-to-4 (itw_generate_mips_device, _srgb, _f16) -- and the save path built on it
(itw_dds_encode_texture, itw_dds_encode_pixels) on real, HDR-special and large content, through every launch path.

Content: the reference's sample images (tests/golden/sample_images.npz) at native size; mosaics of them (128x128 tiles, each
turned by a quarter turn per tile so that no level is periodic) at the sizes where the planner of csrc/itw_mips.inc changes its
choice; a small LDR catalogue (flat, 0/255 checkerboards, one-LSB ramps, lone outliers, alpha-only variation) and a half-domain
catalogue (uniform 16-bit patterns, the special halves -- +-0, denormals, +-65504, +-1 and the exponent-31 patterns 0x7C00,
0x7C01, 0x7E00, 0x7FFF and their negatives --, all-negative and denormal-only input).

CPU: the oracle chains equal the reference's own generator bodies (live from oracle/_ref where it is built, through the stored
digests elsewhere), and the kernels' per-level routines (tests/emu) equal the oracle, on every item.  GPU: every level of the
device chain, padding included, equals the oracle chain padded by edge replication, for each codec at every planner branch, for
padded and offset level-0 layouts, partial chains, a caller stream, inside exactly the scratch itw_mip_scratch_bytes sizes;
rejected arguments launch nothing; the DDS save path equals oracle chain + oracle encode at itw_dds_image_offset.

Half conversion: the front end and the RGBA16F filters use the DirectXMath 3.06 scalar half -> float conversion
(csrc/frontend.cuh), which decodes exponent 31 as an ordinary binade (0x7C00 = 65536, 0x7FFF = 131008).  numpy's float16 reads
those patterns as inf / NaN, so the expectations here go through half_to_float below instead."""
import ctypes
import functools
import zlib

import numpy as np
import pytest

import itw_testlib as T
import test_frontend as FE
import test_gpu_content as GC
import test_mips as LM
import test_mips_f16 as HM

B = T.binding
NORM = B.FRONT_NORMALIZE


def half_to_float(h):
    """DirectXMath 3.06 XMConvertHalfToFloat on an array of half bit patterns: exponent 31 is an ordinary binade."""
    h = np.asarray(h).astype(np.uint32)
    s, e, m = h >> 15, (h >> 10) & 31, h & 0x3FF
    normal = ((s << 31) | ((e + 112) << 23) | (m << 13)).astype(np.uint32).view(np.float32)
    denormal = np.where(s == 1, np.float32(-1), np.float32(1)) * m.astype(np.float32) * np.float32(2.0 ** -24)
    return np.where(e > 0, normal, denormal).astype(np.float32)


def full_levels(w, h):
    return max(w, h).bit_length()


def dims(h, w, l):
    return max(1, h >> l), max(1, w >> l)


# ---------------------------------------------------------------------------------------------
# content: "sample:<name>", "mosaic:<h>x<w>", "cat:<family>:<h>x<w>", "crop:<name>:<y>:<x>:<h>x<w>"
# ---------------------------------------------------------------------------------------------
LDR_FAMILIES = ("flat", "checker", "ramp", "outlier", "alpha")
HDR_FAMILIES = ("random", "specials", "negative", "denormal")
SPECIAL_HALVES = (0x0000, 0x8000, 0x0001, 0x8001, 0x03FF, 0x83FF, 0x0400, 0x8400, 0x3C00, 0xBC00, 0x7BFF, 0xFBFF,
                  0x7C00, 0x7C01, 0x7E00, 0x7FFF, 0xFC00, 0xFC01, 0xFE00, 0xFFFF)
# (h, w): box, linear, wide power of two (integer levels, then stale-tap float levels), tall power of two
LDR_CAT_SIZES = ((64, 64), (37, 61), (16, 128), (128, 16))
# (h, w): box, linear and the stale tap, on both axes
HDR_CAT_SIZES = ((64, 64), (37, 61), (1, 16), (16, 1), (8, 64), (64, 8), (5, 3), (17, 256), (100, 3))
# (h, w): linear filter at large coordinates, one-texel-wide levels, extreme aspect ratios (cheap on CPU)
LDR_LARGE = ((3000, 1000), (2047, 2049), (5, 4097), (16383, 5), (8192, 3), (6, 8192))
HDR_LARGE = ((2047, 2049), (5, 4097))


def _shape(text):
    h, w = text.split("x")
    return int(h), int(w)


def _tiles(hdr):
    names = [n for n in (GC.HDR_SAMPLES if hdr else GC.LDR_SAMPLES) if min(GC.sample(n).shape[:2]) >= 128]
    return [GC.sample(n)[:128, :128] for n in names]


def mosaic(hdr, h, w):
    tiles = _tiles(hdr)
    th, tw = -(-h // 128), -(-w // 128)
    rows = [np.concatenate([np.rot90(tiles[(3 * i + j) % len(tiles)], (i + j) % 4) for j in range(tw)], 1) for i in range(th)]
    return np.ascontiguousarray(np.concatenate(rows, 0)[:h, :w])


def ldr_pattern(fam, h, w):
    y, x = np.mgrid[:h, :w]
    img = np.zeros((h, w, 4), np.int64)
    if fam == "flat":
        img[:] = (37, 200, 91, 255)
    elif fam == "checker":                  # 0 / 255 only: box averages and linear weights meet .5 ties
        c = ((x + y) & 1) * 255
        img[..., 0], img[..., 1] = c, 255 - c
        img[..., 2] = (((x >> 1) + (y >> 1)) & 1) * 255
        img[..., 3] = (x & 1) * 255
    elif fam == "ramp":                     # one-LSB steps
        img[..., 0], img[..., 1] = 100 + (x & 1), 200 + (y & 1)
        img[..., 2] = (x + y) % 256
        img[..., 3] = 254 + ((x >> 1) & 1)
    elif fam == "outlier":                  # flat, with single texels far off on a sparse lattice
        img[:] = (10, 20, 30, 255)
        img[(y % 13 == 5) & (x % 11 == 3)] = (255, 255, 255, 0)
    elif fam == "alpha":                    # colour flat, alpha varies
        img[:] = (128, 64, 32, 0)
        img[..., 3] = (7 * x + 13 * y) % 256
    return img.astype(np.uint8)


def hdr_pattern(fam, h, w):
    rng = np.random.default_rng(zlib.crc32(f"{fam}:{h}x{w}".encode()))
    size = (h, w, 4)
    if fam == "random":
        v = rng.integers(0, 0x10000, size)
    elif fam == "specials":
        v = np.array(SPECIAL_HALVES)[rng.integers(0, len(SPECIAL_HALVES), size)]
    elif fam == "negative":
        v = rng.integers(0x8000, 0x10000, size)
    else:                                   # denormals and zeros of both signs
        v = rng.integers(0, 0x400, size) | (rng.integers(0, 2, size) << 15)
    return v.astype(np.uint16)


@functools.lru_cache(None)
def source(item, hdr):
    kind, _, rest = item.partition(":")
    if kind == "sample":
        return GC.sample(rest)
    if kind == "mosaic":
        return mosaic(hdr, *_shape(rest))
    if kind == "cat":
        fam, size = rest.split(":")
        return (hdr_pattern if hdr else ldr_pattern)(fam, *_shape(size))
    name, y, x, size = rest.split(":")
    h, w = _shape(size)
    return np.ascontiguousarray(GC.sample(name)[int(y):int(y) + h, int(x):int(x) + w])


LDR_ITEMS = ([f"sample:{n}" for n in GC.LDR_SAMPLES] + [f"cat:{f}:{h}x{w}" for f in LDR_FAMILIES for h, w in LDR_CAT_SIZES]
             + [f"mosaic:{h}x{w}" for h, w in LDR_LARGE])
HDR_ITEMS = ([f"sample:{n}" for n in GC.HDR_SAMPLES] + [f"cat:{f}:{h}x{w}" for f in HDR_FAMILIES for h, w in HDR_CAT_SIZES]
             + [f"mosaic:{h}x{w}" for h, w in HDR_LARGE])


def ldr_key(item, srgb):
    return f"prepass:rgba8:{item}:{'srgb' if srgb else 'unorm'}"


def hdr_key(item):
    return f"prepass:f16:{item}"


def oracle_levels(codec, item):
    """The oracle's full chain of an item, unpadded."""
    img = source(item, codec == "f16")
    h, w = img.shape[:2]
    if codec == "f16":
        return HM.oracle_chain(img, full_levels(w, h))
    return T.oracle_mip_chain_rgba8(img, codec == "srgb", pad=False)


@functools.lru_cache(4)
def expected(codec, item):
    """The oracle's full chain padded by edge replication; checked against the stored digest of the reference's chain where
    the CPU tests pin that item (the reference is not read)."""
    chain = oracle_levels(codec, item)
    key = hdr_key(item) if codec == "f16" else ldr_key(item, codec == "srgb")
    if item in (HDR_ITEMS if codec == "f16" else LDR_ITEMS):
        assert T.same(HM.flat(chain), T.reference(key, None)), f"{key}: the oracle differs from the stored reference digest"
    return [HM.pad4(l) for l in chain]


def texel_bits(t):
    return f"{int.from_bytes(np.ascontiguousarray(t).tobytes(), 'little'):0{2 * t.nbytes}x}"


def level_report(what, l, want, got, limit=8):
    """'' when equal; else the number of differing texels of level l and, for the first `limit`, (x, y) and the expected and
    actual texel bits (RGBA8: ABGR as one little-endian word; RGBA16F: four halves, alpha first)."""
    if want.shape != got.shape:
        return f"{what} level {l}: shape {got.shape} instead of {want.shape}"
    bad = (want != got).any(-1)
    if not bad.any():
        return ""
    ys, xs = np.nonzero(bad)
    lines = [f"{what} level {l} ({want.shape[1]}x{want.shape[0]} padded): {ys.size} of {bad.size} texels differ"]
    lines += [f"  ({x}, {y}) expected {texel_bits(want[y, x])}, got {texel_bits(got[y, x])}" for y, x in zip(ys[:limit], xs[:limit])]
    return "\n".join(lines)


# ---------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------
def test_half_to_float_is_the_directxmath_306_conversion():
    """half_to_float over all 65,536 patterns equals the reference's own F16toF32 (live or stored); exponent 31 is a binade
    (where numpy's float16 reads inf / NaN), and the front end's float -> half takes every value back to its pattern."""
    allh = np.arange(0x10000)
    got = half_to_float(allh)
    lib = T.ref_frontend()
    want = T.reference("prepass:half_to_float:all",
                       lib and (lambda: np.array([lib.ref_half_to_float(int(b)) for b in allh], np.float32).view(np.uint32)))
    assert T.same(got.view(np.uint32), want)
    assert (got[0x7C00], got[0x7C01], got[0x7E00], got[0x7FFF], got[0xFC00]) == (65536, 65600, 98304, 131008, -65536)
    assert got[0x8000].view(np.uint32) == 0x80000000 and got[1] == np.float32(2.0 ** -24)
    assert np.isinf(np.array([0x7C00], np.uint16).view(np.float16)[0]) and np.isnan(np.array([0x7E00], np.uint16).view(np.float16)[0])
    back = T.oracle().convert_pixels("BC6H", got.reshape(256, 256, 1), 0, pad=False)[..., 0]
    assert np.array_equal(back.reshape(-1), allh)


def test_catalogues_reach_the_edges():
    for h, w in HDR_CAT_SIZES:
        if h * w >= 64:
            sp = source(f"cat:specials:{h}x{w}", True)
            assert set(SPECIAL_HALVES) <= set(np.unique(sp).tolist()), (h, w)
        assert (source(f"cat:negative:{h}x{w}", True) >= 0x8000).all()
        assert ((source(f"cat:denormal:{h}x{w}", True) & 0x7C00) == 0).all()
    chk = source("cat:checker:37x61", False)
    assert set(np.unique(chk).tolist()) == {0, 255}
    ramp = source("cat:ramp:64x64", False).astype(int)
    assert np.abs(np.diff(ramp[..., 0], axis=1)).max() == 1
    m = source("mosaic:300x400", False)
    assert m.shape == (300, 400, 4) and not np.array_equal(m[:128, :128], m[128:256, 128:256])


@pytest.mark.parametrize("item", LDR_ITEMS)
def test_rgba8_oracle_equals_reference(item):
    """Both RGBA8 codecs: the oracle chain equals the reference's own generator bodies (DirectXTex's box / linear filters)."""
    lib = LM.ref_lib()
    img = source(item, False)
    for srgb in (0, 1):
        want = T.reference(ldr_key(item, srgb), lib and (lambda: LM.flat(LM.chain_with(lib.ref_mip_chain_rgba8, img, srgb))))
        assert T.same(LM.flat(oracle_levels("srgb" if srgb else "unorm", item)), want), (item, srgb)


@pytest.mark.parametrize("item", HDR_ITEMS)
def test_f16_oracle_equals_reference(item):
    lib = T.ref_frontend()
    img = source(item, True)
    levels = full_levels(img.shape[1], img.shape[0])
    want = T.reference(hdr_key(item), lib and (lambda: HM.flat(HM.chain_with(lib.ref_mip_chain_f16, img, levels))))
    assert T.same(HM.flat(oracle_levels("f16", item)), want), item


@pytest.mark.parametrize("item", LDR_ITEMS)
def test_rgba8_emulation_equals_oracle(item):
    """The kernels' per-texel routines (integer box, float filter with the stale row) with the host's per-level choice."""
    img = source(item, False)
    for srgb in (0, 1):
        want = [HM.pad4(l) for l in oracle_levels("srgb" if srgb else "unorm", item)]
        for l, got in enumerate(LM.emulated_chain(img, srgb)):
            assert not (r := level_report(f"emulated {'srgb' if srgb else 'unorm'} {item}", l, want[l], got)), r


@pytest.mark.parametrize("item", HDR_ITEMS)
def test_f16_emulation_equals_oracle(item):
    img = source(item, True)
    want = [HM.pad4(l) for l in oracle_levels("f16", item)]
    for l, got in enumerate(HM.emulated_chain(img, len(want)), 1):
        assert not (r := level_report(f"emulated f16 {item}", l, want[l], got)), r


def test_level_report_names_texels_and_bits():
    want = HM.pad4(source("cat:specials:5x3", True))
    got = want.copy()
    got[1, 2, 0] ^= 0x8000
    got[7, 3] = 0x7C00
    r = level_report("f16 cat:specials:5x3 tight", 2, want, got)
    assert r.startswith("f16 cat:specials:5x3 tight level 2 (4x8 padded): 2 of 32 texels differ"), r
    assert f"(2, 1) expected {texel_bits(want[1, 2])}, got {texel_bits(got[1, 2])}" in r
    assert "got 7c007c007c007c00" in r
    assert level_report("x", 0, want, want) == ""
    many = level_report("x", 0, want, want ^ np.uint16(1))
    assert len(many.splitlines()) == 1 + 8


# unclipped 32-bit sources for the BC6H save path: (name, h, w, planes)
PIXEL_SOURCES = [("specials", 12, 20, 3), ("specials", 16, 32, 4), ("monkey-scaled", 220, 220, 3), ("monkey-scaled", 64, 128, 3)]


@functools.lru_cache(None)
def pixel_source(name, h, w, planes):
    """float32 planes: the front end's special values (inf, NaN, 1e9, 65504 .. 131040, negatives, denormals) in a seeded
    arrangement, or monkey-32bit.hdr scaled so that its brightest texels pass 65504 and 131008 (no clipping)."""
    if name == "specials":
        rng = np.random.default_rng(h * 1000 + w)
        return FE.SPECIALS[rng.integers(0, len(FE.SPECIALS), (h, w, planes))].astype(np.float32)
    f = half_to_float(GC.sample("monkey-32bit.hdr"))[:h, :w, :planes]
    return (f * np.float32(150000.0 / f[..., :3].max())).astype(np.float32)


def pixels_levels(api, px, flags, levels, emulate=False):
    """The save path of itw_dds_encode_pixels for RGBA16F up to the encoder: convert (+flip) -> mip chain -> normalise every
    level -> pad.  The normalise step is `api`'s front end on the level read back through half_to_float (an identity
    conversion under the 3.06 rules).  emulate=True takes the chain from the kernel's per-level routine."""
    top = api.convert_pixels("BC6H", px, flags & ~NORM, pad=False)
    chain = [top] + (HM.emulated_chain(top, levels) if emulate else HM.oracle_chain(top, levels)[1:])
    out = []
    for lv in chain:
        lv = np.ascontiguousarray(lv)
        if flags & NORM:
            rgb = api.convert_pixels("BC6H", half_to_float(lv), NORM, pad=False)
            lv = np.concatenate([rgb[..., :3], lv[..., 3:]], axis=2)
        out.append(HM.pad4(lv))
    return out


@pytest.mark.parametrize("name,h,w,planes", PIXEL_SOURCES)
def test_unclipped_hdr_save_path_emulated(name, h, w, planes):
    """The kernels' front-end and filter routines on unclipped 32-bit sources equal the oracle, level by level."""
    px = pixel_source(name, h, w, planes)
    levels = full_levels(w, h)
    for flags in ((0, NORM, 1) if planes == 4 else (0, NORM)):
        want = pixels_levels(T.oracle(), px, flags, levels)
        got = pixels_levels(T.emu(), px, flags, levels, emulate=True)
        for l in range(levels):
            assert not (r := level_report(f"emulated f16 pixels {name} {w}x{h} flags {flags}", l, want[l], got[l])), r


# ---------------------------------------------------------------------------------------------
# GPU: the device chains
# ---------------------------------------------------------------------------------------------
CODECS = {"unorm": ("itw_generate_mips_device", 4), "srgb": ("itw_generate_mips_device_srgb", 4), "f16": ("itw_generate_mips_device_f16", 8)}
CANARY = 4096
# (h, w) of sample mosaics, by the planner branch they reach (csrc/itw_mips.inc generate_mips_impl)
GPU_SHAPES = [
    (4096, 4096), (2048, 2048),                     # 128-bit integer kernel on the big levels, then mip_tail_kernel
    (64, 4096), (4096, 64), (4, 8192), (8192, 4),   # integer levels, then float levels whose stale row an integer level made
    (2047, 2049), (3000, 1000), (5, 4097), (16383, 5),   # linear filter at large coordinates; one-texel-wide levels
    (1, 1), (2, 2), (1, 2), (2, 1), (3, 3), (64, 2),     # pad-only chains and padded level 0 plus exact levels
]


def gpu_items(codec):
    return [f"mosaic:{h}x{w}" for h, w in GPU_SHAPES] + [f"sample:{n}" for n in (GC.HDR_SAMPLES if codec == "f16" else GC.LDR_SAMPLES)]


def _mips_fn(lib, codec):
    f = getattr(lib.lib, CODECS[codec][0])
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.POINTER(B.RgbaSurface), ctypes.c_int, ctypes.POINTER(B.RgbaSurface), ctypes.c_void_p, ctypes.c_void_p]
    return f


def device_level0(img, extra, offset, texel):
    """img on the device at `offset` bytes into an allocation, rows `extra` bytes apart beyond the texels (filled with 0x5A);
    returns (tensor, pointer, stride).  Runs on the current torch stream."""
    import torch
    h, w = img.shape[:2]
    row, stride = w * texel, w * texel + extra
    host = np.full((h, stride), 0x5A, np.uint8)
    host[:, :row] = np.ascontiguousarray(img).view(np.uint8).reshape(h, row)
    d = torch.empty(offset + h * stride, dtype=torch.uint8, device="cuda")
    d[offset:] = torch.from_numpy(host.reshape(-1)).cuda()
    return d, d.data_ptr() + offset, stride


def run_chain(codec, img, levels, extra=0, offset=0, on_stream=False):
    """One device chain inside exactly itw_mip_scratch_bytes (x2 for RGBA16F) between two 4 KiB canaries of one allocation.
    Checks the canaries and that every produced level lies inside the scratch with stride pw * texel and without overlap;
    returns the levels (None for an unpadded level 0, which is the input itself)."""
    import torch
    lib = T.product()
    texel = CODECS[codec][1]
    h, w = img.shape[:2]
    pad0 = bool((w | h) & 3)
    nbytes = lib.lib.itw_mip_scratch_bytes(w, h, levels, 0 if pad0 else 1) * (2 if codec == "f16" else 1)
    s = torch.cuda.Stream() if on_stream else torch.cuda.current_stream()
    with torch.cuda.stream(s):
        d0, ptr, stride = device_level0(img, extra, offset, texel)
        guard = torch.full((2 * CANARY + nbytes,), 0xA5, dtype=torch.uint8, device="cuda")
        scratch = guard.data_ptr() + CANARY
        top = B.RgbaSurface(ptr, w, h, stride)
        outs = (B.RgbaSurface * levels)()
        rc = _mips_fn(lib, codec)(ctypes.byref(top), levels, outs, ctypes.c_void_p(scratch), ctypes.c_void_p(s.cuda_stream))
        assert rc == 0, lib.last_error()
    s.synchronize()
    g = guard.cpu().numpy()
    assert (g[:CANARY] == 0xA5).all() and (g[CANARY + nbytes:] == 0xA5).all(), f"{codec} {h}x{w}: a canary next to the scratch was overwritten"
    res, spans = [], []
    for l in range(levels):
        dh, dw = dims(h, w, l)
        ph, pw = dh + (-dh) % 4, dw + (-dw) % 4
        o = outs[l]
        if l == 0 and not pad0:
            assert (o.ptr, o.width, o.height, o.stride) == (ptr, w, h, stride), "unpadded level 0 must be the input"
            res.append(None)
            continue
        assert (o.width, o.height, o.stride) == (pw, ph, pw * texel), (l, o.width, o.height, o.stride)
        off, size = (o.ptr or 0) - scratch, ph * pw * texel
        assert 0 <= off and off + size <= nbytes, f"level {l} at scratch offset {off} (+{size}) outside {nbytes} bytes"
        spans.append((off, off + size, l))
        res.append(g[CANARY + off:CANARY + off + size].view(np.uint16 if codec == "f16" else np.uint8).reshape(ph, pw, 4))
    spans.sort()
    for a, b in zip(spans, spans[1:]):
        assert a[1] <= b[0], f"levels {a[2]} and {b[2]} overlap"
    del d0
    return res


def check_chain(codec, item, levels=None, layout="tight", extra=0, offset=0, on_stream=False):
    want = expected(codec, item)
    img = source(item, codec == "f16")
    got = run_chain(codec, img, levels or len(want), extra, offset, on_stream)
    h, w = img.shape[:2]
    for l, g in enumerate(got):
        if g is not None:
            assert not (r := level_report(f"{codec} {item} ({w}x{h}) {layout}, {len(got)} of {len(want)} levels", l, want[l], g)), r


CHAIN_CASES = [(c, i) for c in CODECS for i in gpu_items(c)]


@pytest.mark.gpu
@pytest.mark.parametrize("codec,item", CHAIN_CASES, ids=[f"{c}-{i}" for c, i in CHAIN_CASES])
def test_gpu_chain_every_planner_branch(codec, item):
    """Tight level 0, full chain, default stream."""
    check_chain(codec, item)


LAYOUT_ITEMS = {"unorm": ["sample:baboon.png", "sample:normals.png", "sample:monkey.png", "mosaic:64x4096"],
                "f16": ["sample:HDR.hdr", "sample:monkey-32bit.hdr", "mosaic:64x4096", "mosaic:37x61"]}
LAYOUT_ITEMS["srgb"] = LAYOUT_ITEMS["unorm"]
LAYOUT_CASES = [(c, i) for c in CODECS for i in LAYOUT_ITEMS[c]]


@pytest.mark.gpu
@pytest.mark.parametrize("codec,item", LAYOUT_CASES, ids=[f"{c}-{i}" for c, i in LAYOUT_CASES])
def test_gpu_chain_level0_layouts(codec, item):
    """Padded strides and a level 0 one texel off its allocation: strides that are not multiples of 16 bytes and the offset
    pointer must take the plain kernel for level 1 (128x128: the tail reads the strided level 0) and give identical bytes."""
    texel = CODECS[codec][1]
    extras = (8, 16, 24) if texel == 8 else (4, 12, 16)
    for layout, extra, offset in [("tight", 0, 0)] + [(f"stride+{e}", e, 0) for e in extras] + [("offset+1 texel", 0, texel)]:
        check_chain(codec, item, layout=layout, extra=extra, offset=offset)


CHAIN_ITEMS = {"unorm": ["sample:normals.png", "sample:monkey.png", "mosaic:64x4096", "mosaic:2047x2049", "mosaic:3x3"],
               "f16": ["sample:HDR.hdr", "sample:monkey-32bit.hdr", "mosaic:64x4096", "mosaic:2047x2049", "mosaic:3x3"]}
CHAIN_ITEMS["srgb"] = CHAIN_ITEMS["unorm"]
PARTIAL_CASES = [(c, i) for c in CODECS for i in CHAIN_ITEMS[c]]


@pytest.mark.gpu
@pytest.mark.parametrize("codec,item", PARTIAL_CASES, ids=[f"{c}-{i}" for c, i in PARTIAL_CASES])
def test_gpu_partial_chains(codec, item):
    """levels = 1, 2, 3, full - 1 and full: the tail and the integer-kernel choice are made over the requested levels only."""
    full = len(expected(codec, item))
    for levels in sorted({1, 2, 3, full - 1, full} & set(range(1, full + 1))):
        check_chain(codec, item, levels=levels)


STREAM_ITEMS = {"unorm": ["sample:baboon.png", "mosaic:2048x2048"], "srgb": ["sample:monkey.png", "mosaic:2048x2048"],
                "f16": ["sample:HDR.hdr", "mosaic:2048x2048"]}
STREAM_CASES = [(c, i) for c in CODECS for i in STREAM_ITEMS[c]]


@pytest.mark.gpu
@pytest.mark.parametrize("codec,item", STREAM_CASES, ids=[f"{c}-{i}" for c, i in STREAM_CASES])
def test_gpu_chain_on_caller_stream(codec, item):
    """Level 0 produced on a non-default stream and the chain enqueued on that stream (and a padded stride)."""
    check_chain(codec, item, layout="caller stream", on_stream=True)
    check_chain(codec, item, layout="caller stream, stride+16", extra=16, on_stream=True)


@pytest.mark.gpu
@pytest.mark.parametrize("codec", list(CODECS))
def test_gpu_rejected_arguments(codec):
    """Each must return non-zero with an error text and launch nothing; the largest accepted height works."""
    import torch
    lib = T.product()
    f = _mips_fn(lib, codec)
    texel = CODECS[codec][1]
    d = torch.zeros(64 * 64 * texel + 64, dtype=torch.uint8, device="cuda")
    scratch = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    p, sp = d.data_ptr(), scratch.data_ptr()
    cases = [("pointer not aligned to the texel", p + texel // 2, 64, 64, 64 * texel, 7, sp),
             ("stride not aligned to the texel", p, 60, 60, 60 * texel + texel // 2, 6, sp),
             ("stride smaller than a row", p, 64, 64, 63 * texel, 7, sp),
             ("null scratch, levels > 1", p, 64, 64, 64 * texel, 2, None),
             ("null scratch, level 0 to pad", p, 62, 64, 62 * texel, 1, None),
             ("height 65533", p, 4, 65533, 4 * texel, 1, sp)]
    torch.cuda.synchronize()
    for what, ptr, w, h, stride, levels, scr in cases:
        outs = (B.RgbaSurface * levels)()
        before = lib.launch_count()
        rc = f(ctypes.byref(B.RgbaSurface(ptr, w, h, stride)), levels, outs, ctypes.c_void_p(scr), None)
        assert rc != 0, what
        assert lib.last_error(), what
        assert lib.launch_count() == before, f"{what}: launched a kernel"
    check_chain(codec, "mosaic:65532x4")


# ---------------------------------------------------------------------------------------------
# GPU: the save path
# ---------------------------------------------------------------------------------------------
def _crops(name, n, size):
    h, w = size
    img = GC.sample(name)
    return [f"crop:{name}:{(37 * i) % (img.shape[0] - h)}:{(53 * i + 11) % (img.shape[1] - w)}:{h}x{w}" for i in range(n)]


# id: (dxgi, profile, items, placement per item (h host, d device), extra stride bytes, cube)
SAVE_CASES = {
    "bc1-monkey-host-padded": (71, None, ["sample:monkey.png"], "h", 12, 0),
    "bc1srgb-normals-device-padded": (72, None, ["sample:normals.png"], "d", 16, 0),
    "bc3-array3-mixed": (77, None, ["sample:baboon.png", "sample:juggling-balls.jpg", "sample:colors-260K.png"], "hdh", 4, 0),
    "bc3srgb-monkey-device": (78, None, ["sample:monkey.png"], "d", 0, 0),
    "bc4-gradients-host": (80, None, ["sample:gradients.png"], "h", 0, 0),
    "bc5-normals-device-padded": (83, None, ["sample:normals.png"], "d", 64, 0),
    "bc7-colors16M-host-padded": (98, "fast", ["sample:colors-16M.png"], "h", 4, 0),
    "bc7srgb-256-mixed": (99, "fast", ["sample:radial-grayscale.png", "sample:gradients.png"], "dh", 8, 0),
    "bc3-two-cubes-17-mixed": (77, None, _crops("monkey.png", 12, (17, 17)), "hd" * 6, 4, 1),
    "bc6h-hdr-device-padded": (95, "bc6h_veryfast", ["sample:HDR.hdr"], "d", 24, 0),
    "bc6h-sf16-monkey-host-padded": (96, "bc6h_fast", ["sample:monkey-32bit.hdr"], "h", 8, 0),
    "bc6h-cube-24-mixed": (95, "bc6h_veryfast", _crops("HDR.hdr", 3, (24, 24)) + _crops("monkey-32bit.hdr", 3, (24, 24)), "hdhdhd", 16, 1),
}
SRGB_DXGI = (72, 78, 99)


def _format_name(dxgi):
    return {71: "BC1", 72: "BC1", 77: "BC3", 78: "BC3", 80: "BC4", 83: "BC5", 95: "BC6H", 96: "BC6H", 98: "BC7", 99: "BC7"}[dxgi]


def check_blob(lib, desc, blob, per_item_levels, fmt, prof, what):
    """Every level of every item at itw_dds_image_offset equals the oracle's encoding of the expected padded level."""
    o = T.oracle()
    s = o.profile(prof) if prof else None
    hdr = lib.lib.itw_dds_header_bytes(ctypes.byref(desc))
    assert sum(lib.lib.itw_dds_image_bytes(ctypes.byref(desc), m) for m in range(desc.mip_levels)) * desc.array_size == blob.size - hdr
    bpb = B.FORMATS[fmt][1]
    for item, levels in enumerate(per_item_levels):
        for mip, lv in enumerate(levels):
            want = o.encode(fmt, np.ascontiguousarray(lv), s)
            off = lib.lib.itw_dds_image_offset(ctypes.byref(desc), item, mip)
            got = blob[off:off + want.size]
            assert np.array_equal(got, want), (f"{what}: item {item} level {mip} ({lv.shape[1]}x{lv.shape[0]}): "
                                               f"{T.differing_blocks(got, want, bpb)} of {want.size // bpb} blocks differ")


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SAVE_CASES))
def test_gpu_encode_texture_equals_oracle_chain_and_encode(case):
    """itw_dds_encode_texture: host and device level-0 surfaces (padded strides, mixed in one call), arrays, cube maps,
    an odd size with several items (per-item scratch off 16-byte alignment) == oracle chain + pad + oracle encode."""
    import torch
    dxgi, prof, items, placement, extra, cube = SAVE_CASES[case]
    fmt = _format_name(dxgi)
    hdr = fmt == "BC6H"
    texel = 8 if hdr else 4
    lib = T.product()
    imgs = [source(i, hdr) for i in items]
    h, w = imgs[0].shape[:2]
    levels = full_levels(w, h)
    keep, surfaces = [], []
    for img, where in zip(imgs, placement):
        if where == "d":
            d, ptr, stride = device_level0(img, extra, 0, texel)
            keep.append(d)
        else:
            host = np.full((h, w * texel + extra), 0x5A, np.uint8)
            host[:, :w * texel] = img.view(np.uint8).reshape(h, w * texel)
            keep.append(host)
            ptr, stride = host.ctypes.data, host.strides[0]
        surfaces.append(B.RgbaSurface(ptr, w, h, stride))
    torch.cuda.synchronize()
    desc = B.DdsDesc(w, h, levels, len(items), dxgi, cube)
    n = lib.lib.itw_dds_file_bytes(ctypes.byref(desc))
    blob = np.zeros(n, np.uint8)
    settings = lib.profile(prof) if prof else None
    sp = ctypes.cast(ctypes.byref(settings), ctypes.c_void_p) if settings is not None else None
    got = lib.lib.itw_dds_encode_texture(ctypes.byref(desc), (B.RgbaSurface * len(surfaces))(*surfaces), sp, blob.ctypes.data, n)
    assert got == n, lib.last_error()
    codec = "f16" if hdr else ("srgb" if dxgi in SRGB_DXGI else "unorm")
    per_item = [[HM.pad4(l) for l in oracle_levels(codec, i)] for i in items]
    check_blob(lib, desc, blob, per_item, fmt, prof, f"{case} ({', '.join(items[:3])}{' ...' if len(items) > 3 else ''})")


PIXEL_CASES = [(dxgi, src, flags) for src in PIXEL_SOURCES for dxgi, flags in ((95, 0), (96, NORM))]
PIXEL_CASES += [(95, PIXEL_SOURCES[1], 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("dxgi,src,flags", PIXEL_CASES, ids=[f"{d}-{s[0]}-{s[1]}x{s[2]}x{s[3]}-f{f}" for d, s, f in PIXEL_CASES])
def test_gpu_encode_pixels_unclipped_bc6h(dxgi, src, flags):
    """itw_dds_encode_pixels from unclipped 32-bit planes (values past 65504 become exponent-31 halves that the chain and the
    normalise step read as 65536 .. 131008) == oracle convert -> chain -> normalise (through half_to_float) -> pad -> encode."""
    lib = T.product()
    px = pixel_source(*src)
    h, w = px.shape[:2]
    levels = full_levels(w, h)
    desc = B.DdsDesc(w, h, levels, 1, dxgi, 0)
    prof = "bc6h_veryfast"
    blob = lib.dds_encode_pixels(desc, [px], flags, lib.profile(prof))
    want = pixels_levels(T.oracle(), px, flags, levels)
    check_blob(lib, desc, blob, [want], "BC6H", prof, f"{dxgi} pixels {src[0]} {w}x{h}x{src[3]} flags {flags}")


@pytest.mark.gpu
def test_gpu_encode_texture_fanned_out_over_devices():
    """save_texture_fanout (>= 2^20 texels, host level 0) over every visible GPU gives the single-device file."""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"fan-out over devices needs two or more visible GPUs; {n} visible")
    lib = T.product()
    img = source("mosaic:1024x2048", False)
    desc = B.DdsDesc(2048, 1024, full_levels(2048, 1024), 1, 71, 0)
    one = lib.dds_encode_texture(desc, [img])
    lib.set_devices(list(range(n)))
    try:
        many = lib.dds_encode_texture(desc, [img])
    finally:
        lib.set_devices([])
    assert np.array_equal(many, one), f"{T.differing_blocks(many, one, 8)} blocks differ"
