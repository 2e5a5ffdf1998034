"""RGBA16F mip chain of the BC6H save path (include/itw_bcn.h, itw_generate_mips_device_f16).

For BC6H the plug-in forces DirectXTex's own (non-WIC) generator, whose code is in the reference tree.  CPU: (1) the
oracle restatement (oracle/itw_oracle_frontend.cpp, oracle_mip_chain_f16) against the reference's OWN
_Generate2DMipsBoxFilter / _Generate2DMipsLinearFilter bodies (oracle/_ref/libitw_ref_frontend.so); (2) the kernel's
per-texel routine (csrc/mips_f16.cuh through tests/emu) against the oracle, including the stale fourth tap of wide
power-of-two textures.  GPU: the device chain and the BC6H DDS save path against the oracle."""
import ctypes

import numpy as np
import pytest

import itw_testlib as T

D = T.binding.DdsDesc
SIZES = [(64, 64), (8, 64), (64, 8), (1, 16), (16, 1), (2, 32), (4, 4), (1, 1), (27, 50), (5, 3), (3, 100), (100, 3), (1, 9), (48, 64)]


def full_levels(w, h):
    n, m = 1, max(w, h)
    while m > 1:
        m >>= 1
        n += 1
    return n


def level_dims(w, h, levels):
    return [(max(1, h >> l), max(1, w >> l)) for l in range(levels)]


def random_f16(h, w, seed):
    rng = np.random.default_rng(seed)
    img = (rng.random((h, w, 4), dtype=np.float32) * np.float32(200.0)).astype(np.float16)
    img[rng.random((h, w)) < 0.1] = np.float16(0.0)
    img.reshape(-1)[:6] = np.array([65504.0, 6.1e-5, 5.96e-8, 1.0, 0.333, 1000.5], np.float16)[: img.size][:6] if img.size >= 6 else img.reshape(-1)[:6]
    return img.view(np.uint16)


def chain_with(fn, img, levels):
    h, w = img.shape[:2]
    dims = level_dims(w, h, levels)
    out = np.zeros(sum(a * b * 4 for a, b in dims), np.uint16)
    src = np.ascontiguousarray(img)
    assert fn(src.ctypes.data_as(ctypes.c_void_p), w, h, levels, out.ctypes.data_as(ctypes.c_void_p)) == 0
    res, off = [], 0
    for a, b in dims:
        res.append(out[off:off + a * b * 4].reshape(a, b, 4))
        off += a * b * 4
    return res


def flat(chain):
    return np.concatenate([l.reshape(-1) for l in chain])


def oracle_chain(img, levels):
    return chain_with(T.oracle().lib.oracle_mip_chain_f16, img, levels)


def pad4(level):
    h, w = level.shape[:2]
    return np.pad(level, ((0, (-h) % 4), (0, (-w) % 4), (0, 0)), mode="edge")


@pytest.mark.parametrize("h,w", SIZES)
def test_oracle_matches_reference_generators(h, w):
    lib = T.ref_frontend()
    img = random_f16(h, w, seed=h * 131 + w)
    levels = full_levels(w, h)
    want = T.reference(f"mip_chain_f16:{h}x{w}", lib and (lambda: flat(chain_with(lib.ref_mip_chain_f16, img, levels))))
    got = oracle_chain(img, levels)
    assert T.same(flat(got), want)


def emulated_chain(img, levels):
    """The kernel's per-texel routine level by level, with the host's rule for the stale row (csrc/itw_mips.inc:
    generate_mips_impl).  Returns levels 1.. (level 0 is the input), each padded to multiples of 4."""
    emu = T.emu().lib
    h, w = img.shape[:2]
    box = (w & (w - 1)) == 0 and (h & (h - 1)) == 0
    cur = np.ascontiguousarray(img)
    stale_keep, stale_ptr = None, None
    out = []
    for l in range(1, levels):
        dh, dw = max(1, h >> l), max(1, w >> l)
        ph, pw = dh + (-dh) % 4, dw + (-dw) % 4
        got = np.zeros((ph, pw, 4), np.uint16)
        if cur.shape[0] > 1:                                   # the host code's rule for the stale row (itw_mips.inc)
            stale_keep = cur
            stale_ptr = cur.ctypes.data + (cur.shape[0] - 1) * cur.strides[0]
        emu.emu_mip_level_f16(ctypes.c_void_p(cur.ctypes.data), cur.shape[1], cur.shape[0], cur.strides[0], got.ctypes.data_as(ctypes.c_void_p),
                              dw, dh, pw, ph, 1 if box else 0, ctypes.c_void_p(stale_ptr))
        out.append(got)
        cur = np.ascontiguousarray(got[:dh, :dw])
    del stale_keep
    return out


@pytest.mark.parametrize("h,w", SIZES)
def test_emulated_kernel_matches_oracle(h, w):
    img = random_f16(h, w, seed=h * 17 + w)
    levels = full_levels(w, h)
    want = oracle_chain(img, levels)
    for l, got in enumerate(emulated_chain(img, levels), 1):
        assert np.array_equal(got, pad4(want[l])), (l,) + want[l].shape[:2]


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(256, 256), (16, 128), (128, 16), (37, 61), (4, 4), (1, 16), (64, 200)])
def test_gpu_chain_matches_oracle(h, w):
    import torch
    lib = T.product()
    img = random_f16(h, w, seed=h + w)
    levels = full_levels(w, h)
    want = oracle_chain(img, levels)
    d_img = torch.from_numpy(img.view(np.int16).reshape(-1)).cuda()
    pad0 = (w % 4 != 0) or (h % 4 != 0)
    nbytes = 2 * lib.lib.itw_mip_scratch_bytes(w, h, levels, 0 if pad0 else 1)
    scratch = torch.zeros(max(nbytes, 32), dtype=torch.uint8, device="cuda")
    outs = (T.binding.RgbaSurface * levels)()
    top = T.binding.RgbaSurface(d_img.data_ptr(), w, h, w * 8)
    f = lib.lib.itw_generate_mips_device_f16
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.POINTER(T.binding.RgbaSurface), ctypes.c_int, ctypes.POINTER(T.binding.RgbaSurface), ctypes.c_void_p, ctypes.c_void_p]
    assert f(ctypes.byref(top), levels, outs, ctypes.c_void_p(scratch.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    torch.cuda.synchronize()
    base, host = scratch.data_ptr(), scratch.cpu().numpy()
    for l in range(levels):
        if l == 0 and not pad0:
            continue
        expect = pad4(want[l])
        ph, pw = expect.shape[:2]
        assert (outs[l].width, outs[l].height, outs[l].stride) == (pw, ph, pw * 8)
        off = outs[l].ptr - base
        got = host[off:off + ph * pw * 8].view(np.uint16).reshape(ph, pw, 4)
        assert np.array_equal(got, expect), l


@pytest.mark.gpu
def test_gpu_bc6h_texture_save_path():
    """itw_dds_encode_texture for BC6H: RGBA16F level 0 in, .dds out == oracle chain + pad + per-level encodes."""
    lib = T.product()
    for (w, h, items, cube) in ((64, 64, 1, 0), (60, 36, 1, 0), (32, 32, 6, 1), (64, 16, 1, 0)):
        tops = [random_f16(h, w, seed=40 + s) & np.uint16(0x7FFF) for s in range(items)]
        levels = full_levels(w, h)
        d = D(w, h, levels, items, 95, cube)
        s = lib.profile("bc6h_veryfast")
        blob = lib.dds_encode_texture(d, tops, s)
        for item in range(items):
            chain = oracle_chain(tops[item], levels)
            for mip in range(levels):
                off = lib.lib.itw_dds_image_offset(ctypes.byref(d), item, mip)
                want = lib.encode("BC6H", np.ascontiguousarray(pad4(chain[mip])), s)
                assert np.array_equal(blob[off:off + want.size], want), (item, mip)


def test_oracle_matches_committed_reference_digests():
    import hashlib
    import json
    import os
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "frontend_digests.json")))["mip_chain_f16"]
    assert len(golden) == len(SIZES)
    for h, w in SIZES:
        img = random_f16(h, w, seed=h * 131 + w)
        chain = oracle_chain(img, full_levels(w, h))
        assert hashlib.sha256(b"".join(l.tobytes() for l in chain)).hexdigest() == golden[f"{h}x{w}"], (h, w)
