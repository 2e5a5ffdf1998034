"""On-GPU pre-pass (SURVEY.md 8f-2, include/itw_bcn.h section 4): RGBA8 mip chain + pad-to-4.

Contract = DirectXTex's own non-WIC generators (_Generate2DMipsBoxFilter / _Generate2DMipsLinearFilter,
DirectXTexMipmaps.cpp:715-905) on R8G8B8A8_UNORM and -- for *_SRGB encodings, as the plug-in does -- R8G8B8A8_UNORM_SRGB.
CPU: (1) the oracle restatement (oracle_mip_chain_rgba8) against the reference's OWN function bodies cut by
oracle/build_ref_frontend.py, and against their committed digests; (2) the integer 2x2 box (a+b+c+d+2)>>2 of csrc/mips.cuh IS
that float box filter on exact 2:1 levels; (3) the kernels' per-texel routines (tests/emu) against the oracle, with the host's
per-level choice between the integer and the float kernel; (4) the generated sRGB tables against the oracle's functions.
GPU: the device chains and the DDS save path against the oracle."""
import ctypes
import hashlib
import json
import os

import numpy as np
import pytest

import itw_testlib as T

D = T.binding.DdsDesc
SIZES = [(64, 64), (8, 64), (64, 8), (1, 16), (16, 1), (2, 32), (4, 4), (1, 1), (27, 50), (5, 3), (3, 100), (100, 3), (1, 9), (48, 64), (128, 128)]


def full_levels(w, h):
    return max(w, h).bit_length()


def random_rgba8(h, w):
    return np.random.default_rng(h * 1000 + w).integers(0, 256, (h, w, 4), dtype=np.uint8)


def chain_with(fn, img, srgb):
    h, w = img.shape[:2]
    levels = full_levels(w, h)
    dims = [(max(1, h >> l), max(1, w >> l)) for l in range(levels)]
    out = np.zeros(sum(a * b * 4 for a, b in dims), np.uint8)
    src = np.ascontiguousarray(img)
    assert fn(src.ctypes.data, w, h, levels, srgb, out.ctypes.data) == 0
    res, off = [], 0
    for a, b in dims:
        res.append(out[off:off + a * b * 4].reshape(a, b, 4))
        off += a * b * 4
    return res


def ref_lib():
    """The reference's own generators, or None where they are not built."""
    lib = T.ref_frontend()
    if lib is None:
        return None
    lib.ref_mip_chain_rgba8.restype = ctypes.c_int
    lib.ref_mip_chain_rgba8.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    return lib


def flat(chain):
    return np.concatenate([l.reshape(-1) for l in chain])


@pytest.mark.parametrize("h,w", SIZES)
def test_oracle_matches_reference_generators(h, w):
    lib = ref_lib()
    img = random_rgba8(h, w)
    for srgb in (0, 1):
        want = T.reference(f"mip_chain_rgba8:{h}x{w}:{srgb}", lib and (lambda: flat(chain_with(lib.ref_mip_chain_rgba8, img, srgb))))
        got = T.oracle_mip_chain_rgba8(img, srgb, pad=False)
        assert T.same(flat(got), want), srgb


def test_oracle_matches_committed_reference_digests():
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "frontend_digests.json")))["mip_chain_rgba8"]
    assert len(golden) == 2 * len(SIZES)
    for h, w in SIZES:
        img = random_rgba8(h, w)
        for srgb in (0, 1):
            chain = T.oracle_mip_chain_rgba8(img, srgb, pad=False)
            assert hashlib.sha256(b"".join(l.tobytes() for l in chain)).hexdigest() == golden[f"{h}x{w}:{'srgb' if srgb else 'unorm'}"], (h, w, srgb)


def test_integer_box_is_the_float_box_on_exact_levels():
    """csrc/mips.cuh's (a+b+c+d+2)>>2 against AVERAGE4 on byte/255 floats stored with round-to-nearest: 10^7 random quads (a
    quarter of them exact .5 ties), and whole chains of power-of-two textures against the oracle."""
    rng = np.random.default_rng(1)
    q = rng.integers(0, 256, (10_000_000, 4)).astype(np.uint8)
    f = q.astype(np.float32) * np.float32(1 / 255)
    v = (((f[:, 0] + f[:, 1]) + f[:, 2]) + f[:, 3]) * np.float32(0.25)
    out = (np.clip(v, 0, 1) * np.float32(255) + np.float32(0.5)).astype(np.int32)
    assert np.array_equal(out, (q.astype(np.int32).sum(1) + 2) >> 2)
    for n in (64, 256):
        img = random_rgba8(n, n)
        want = T.oracle_mip_chain_rgba8(img, 0, pad=False)
        cur = img
        for l in range(1, len(want)):
            cur = T.synth.box_mip(cur)
            assert np.array_equal(cur, want[l]), (n, l)


def emulated_chain(img, srgb):
    """The kernels' per-texel routines with the host's per-level kernel choice (csrc/itw_mips.inc: generate_mips_impl)."""
    emu = T.emu().lib
    h, w = img.shape[:2]
    levels = full_levels(w, h)
    box = (w & (w - 1)) == 0 and (h & (h - 1)) == 0
    cur = np.ascontiguousarray(img)
    out = [T.synth.pad_to_4(cur)]
    keep, stale_ptr = None, None
    for l in range(1, levels):
        dh, dw = max(1, h >> l), max(1, w >> l)
        ph, pw = dh + (-dh) % 4, dw + (-dw) % 4
        got = np.zeros((ph, pw, 4), np.uint8)
        exact = (not srgb) and box and cur.shape[1] == 2 * dw and cur.shape[0] == 2 * dh
        if cur.shape[0] > 1:
            keep = cur
            stale_ptr = cur.ctypes.data + (cur.shape[0] - 1) * cur.strides[0]
        if exact:
            emu.emu_mip_level(ctypes.c_void_p(cur.ctypes.data), cur.shape[1], cur.shape[0], cur.strides[0], ctypes.c_void_p(got.ctypes.data), dw, dh, pw, ph)
        else:
            emu.emu_mip_level_rgba8(2 if srgb else 1, ctypes.c_void_p(cur.ctypes.data), cur.shape[1], cur.shape[0], cur.strides[0],
                                    ctypes.c_void_p(got.ctypes.data), dw, dh, pw, ph, 1 if box else 0, ctypes.c_void_p(stale_ptr))
        out.append(got)
        cur = np.ascontiguousarray(got[:dh, :dw])
    return out


@pytest.mark.parametrize("h,w", SIZES)
def test_emulated_kernels_match_oracle(h, w):
    img = random_rgba8(h, w)
    for srgb in (0, 1):
        want = T.oracle_mip_chain_rgba8(img, srgb)
        got = emulated_chain(img, srgb)
        for l in range(len(want)):
            assert np.array_equal(got[l], want[l]), (srgb, l)


def test_srgb_tables_match_the_oracle_functions():
    """csrc/srgb_tables.cuh (tools/gen_srgb_tables.py) against oracle_srgb_to_linear / oracle_linear_to_srgb8, through the kernel's own
    routines: every byte, every threshold and its neighbours, and a dense sweep of [0, 1]."""
    o = T.oracle().lib
    o.oracle_srgb_to_linear.restype = ctypes.c_float
    o.oracle_srgb_to_linear.argtypes = [ctypes.c_float]
    o.oracle_linear_to_srgb8.restype = ctypes.c_int
    o.oracle_linear_to_srgb8.argtypes = [ctypes.c_float]
    src = open(os.path.join(T.ROOT, "intel-texture-works-plugin_b200", "csrc", "srgb_tables.cuh")).read()
    import re
    hexes = lambda text: [int(x, 16) for x in re.findall(r"0x([0-9A-F]{8})u", text)]
    to_lin = hexes(src.split("ITW_TABLE_INIT_linear_threshold")[0])
    thr = hexes(src.split("ITW_TABLE_INIT_linear_threshold")[1].split("ITW_TABLE_INIT_linear_base")[0])
    base_words = hexes(src.split("ITW_TABLE_INIT_linear_base")[1])
    first_exp = int(re.search(r"ITW_SRGB_BASE_FIRST_EXP (\d+)", src).group(1))
    assert len(to_lin) == 256 and len(thr) == 255 and len(base_words) == int(re.search(r"ITW_SRGB_BASE_WORDS (\d+)", src).group(1))
    for b in range(256):
        s = np.float32(b) * np.float32(1.0 / 255.0)
        assert np.float32(o.oracle_srgb_to_linear(float(s))).view(np.uint32) == to_lin[b], b
    thr_arr = np.array(thr, np.uint32)

    def table_byte(bits):
        """the kernel's two-level lookup (csrc/mips_f16.cuh mip_srgb8_store), restated on the parsed tables"""
        if bits < (first_exp << 23):
            return 0
        bucket = (bits >> 15) - (first_exp << 8)
        base = (base_words[bucket >> 2] >> (8 * (bucket & 3))) & 255
        got = base + (1 if base < 255 and thr[base] <= bits else 0)
        assert got == int(np.searchsorted(thr_arr, np.uint32(bits), side="right"))        # == the plain count of thresholds
        return got
    probes = set()
    for t in thr:
        probes.update((t - 1, t, t + 1))
    probes.update(np.linspace(0, 0x3F800000, 200001).astype(np.uint32).tolist())
    for bits in probes:
        v = float(np.array([bits], np.uint32).view(np.float32)[0])
        assert table_byte(bits) == o.oracle_linear_to_srgb8(v), hex(bits)


def gpu_chain(lib, img, srgb):
    import torch
    h, w = img.shape[:2]
    levels = full_levels(w, h)
    d_img = torch.from_numpy(img.reshape(-1)).cuda()
    pad0 = (w % 4 != 0) or (h % 4 != 0)
    nbytes = lib.lib.itw_mip_scratch_bytes(w, h, levels, 0 if pad0 else 1)
    scratch = torch.zeros(max(nbytes, 16), dtype=torch.uint8, device="cuda")
    outs = (T.binding.RgbaSurface * levels)()
    top = T.binding.RgbaSurface(d_img.data_ptr(), w, h, w * 4)
    f = lib.lib.itw_generate_mips_device_srgb if srgb else lib.lib.itw_generate_mips_device
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.POINTER(T.binding.RgbaSurface), ctypes.c_int, ctypes.POINTER(T.binding.RgbaSurface), ctypes.c_void_p, ctypes.c_void_p]
    rc = f(ctypes.byref(top), levels, outs, ctypes.c_void_p(scratch.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    lib.check()
    assert rc == 0
    torch.cuda.synchronize()
    base, host = scratch.data_ptr(), scratch.cpu().numpy()
    res = []
    for l in range(levels):
        if l == 0 and not pad0:
            res.append(img)
            continue
        pw, ph = outs[l].width, outs[l].height
        assert outs[l].stride == pw * 4
        off = outs[l].ptr - base
        res.append(host[off:off + ph * pw * 4].reshape(ph, pw, 4))
    return res, nbytes


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(256, 256), (64, 200), (37, 61), (4, 4), (1, 16), (16, 256), (256, 16), (1024, 1024)])
def test_gpu_mip_chain_matches_oracle(h, w):
    lib = T.product()
    img = random_rgba8(h, w)
    for srgb in (0, 1):
        want = T.oracle_mip_chain_rgba8(img, srgb)
        got, nbytes = gpu_chain(lib, img, srgb)
        pad0 = (w % 4 != 0) or (h % 4 != 0)
        assert nbytes == sum(x.size for x in want[(0 if pad0 else 1):])
        for l in range(len(want)):
            assert np.array_equal(got[l], want[l]), (srgb, l)


@pytest.mark.gpu
def test_whole_texture_save_path():
    """itw_dds_encode_texture: level 0 in, .dds out (mips made and encoded on the GPU) == oracle chain + per-level encodes; the
    *_SRGB formats (72 / 78 / 99) take the sRGB-correct chain, as the plug-in does (IntelPlugin.cpp:152-154)."""
    lib = T.product()
    for (w, h, fmt, name, prof, items, cube) in ((128, 64, 77, "BC3", None, 1, 0), (60, 36, 98, "BC7", "veryfast", 1, 0), (32, 32, 71, "BC1", None, 6, 1),
                                                 (64, 64, 72, "BC1", None, 1, 0), (40, 24, 78, "BC3", None, 1, 0), (64, 32, 99, "BC7", "veryfast", 1, 0)):
        tops = [T.synth.mixed_rgba8(h, w, seed=s) for s in range(items)]
        levels = full_levels(w, h)
        d = D(w, h, levels, items, fmt, cube)
        s = lib.profile(prof) if prof else None
        blob = lib.dds_encode_texture(d, tops, s)
        for item in range(items):
            chain = T.oracle_mip_chain_rgba8(tops[item], 1 if fmt in (72, 78, 99) else 0)
            for mip in range(levels):
                off = lib.lib.itw_dds_image_offset(ctypes.byref(d), item, mip)
                want = lib.encode(name, np.ascontiguousarray(chain[mip]), s)
                assert np.array_equal(blob[off:off + want.size], want), (fmt, item, mip)
