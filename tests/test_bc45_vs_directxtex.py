"""BC4 / BC5: the oracle (oracle/itw_oracle.cpp, restated from DirectXTex) against DirectXTex's OWN encoder bodies
(BC4BC5.cpp's namespace body + BC.h's OptimizeAlpha, cut by oracle/build_ref_frontend.py).  Texel floats are
byte * (1/255) (rule F7: in the reference they come from XMLoadUByteN4, DirectXMath, outside the tree).
Also checks the integer decode formula of csrc/decode.cuh against DirectXTex's float decode under round-to-nearest."""
import ctypes
import hashlib
import json
import os

import numpy as np
import pytest

import itw_testlib as T


def ref_lib():
    """DirectXTex's own BC4 / BC5 bodies, or None where they are not built."""
    lib = T.ref_frontend()
    if lib is None:
        return None
    lib.ref_encode_bc4u.restype = None
    lib.ref_encode_bc4u.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.ref_encode_bc5u.restype = None
    lib.ref_encode_bc5u.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.ref_decode_bc4u.restype = None
    lib.ref_decode_bc4u.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    return lib


def ref_encode(lib, fmt, img):
    h, w = img.shape[:2]
    out = []
    scale = np.float32(1.0) / np.float32(255.0)
    for by in range(h // 4):
        for bx in range(w // 4):
            blk = img[4 * by:4 * by + 4, 4 * bx:4 * bx + 4].reshape(16, 4)
            r = np.ascontiguousarray(blk[:, 0].astype(np.float32) * scale)
            g = np.ascontiguousarray(blk[:, 1].astype(np.float32) * scale)
            o = np.zeros(8 if fmt == "BC4" else 16, np.uint8)
            if fmt == "BC4":
                lib.ref_encode_bc4u(r.ctypes.data, o.ctypes.data)
            else:
                lib.ref_encode_bc5u(r.ctypes.data, g.ctypes.data, o.ctypes.data)
            out.append(o)
    return np.concatenate(out)


def adversarial(seed):
    """Blocks that exercise both ramps: touching 0 / 255, flat, two-valued, narrow ranges, random."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (64, 64, 4), dtype=np.uint8)
    img[0:8] = rng.integers(0, 4, (8, 64, 4), dtype=np.uint8)                     # near 0
    img[8:16] = 255 - rng.integers(0, 4, (8, 64, 4), dtype=np.uint8)              # near 255
    img[16:20] = 128                                                               # flat
    img[20:24] = np.where(rng.random((4, 64, 4)) < 0.5, 0, 255).astype(np.uint8)   # two-valued at the extremes
    img[24:32] = (100 + rng.integers(0, 3, (8, 64, 4))).astype(np.uint8)           # narrow
    img[32:36, :, 0] = 0
    img[36:40, :, 0] = 255
    ramp = (np.arange(64, dtype=np.uint32) * 4).astype(np.uint8)
    img[40:44, :, 0] = ramp[None, :]                                               # includes 0 and 252
    return img


@pytest.mark.parametrize("fmt", ["BC4", "BC5"])
def test_oracle_equals_directxtex_encoder_bodies(fmt):
    lib, o = ref_lib(), T.oracle()
    images = dict(T.corpus8())
    images["adversarial1"] = adversarial(1)
    images["adversarial2"] = adversarial(2)
    for name, img in images.items():
        want = T.reference(f"bc45:{fmt}:{name}", lib and (lambda: ref_encode(lib, fmt, img)))
        got = T.run(o, fmt, img, None)
        assert T.same(got, want), (fmt, name) + (() if isinstance(want, str) else (T.differing_blocks(got, want, 8),))


def test_integer_decode_equals_directxtex_float_decode_rounded_to_nearest():
    """csrc/decode.cuh: ((8-q)a0 + (q-1)a1 + 3)/7 etc. == round(255 * DirectXTex's float palette) for every endpoint pair
    and index -- the store to UNORM8 (XMStoreUByteN4) is DirectXMath; round-to-nearest is its documented behaviour."""
    lib = ref_lib()
    import bcn_decode as D
    idx = 0
    for k in range(16):
        idx |= (k % 8) << (3 * k)
    blocks = np.zeros((256 * 256, 8), np.uint8)
    blocks[:, 0] = np.arange(256 * 256) >> 8                   # a0
    blocks[:, 1] = np.arange(256 * 256) & 255                  # a1
    blocks[:, 2:8] = np.frombuffer(int(idx).to_bytes(6, "little"), np.uint8)

    def ref_rounded():
        out = np.zeros((blocks.shape[0], 16), np.float32)
        for blk, o in zip(blocks, out):
            lib.ref_decode_bc4u(np.ascontiguousarray(blk).ctypes.data, o.ctypes.data)
        return np.floor(out.astype(np.float64) * 255.0 + 0.5).astype(np.int64)
    want = T.reference("bc4_decode_rounded:all_endpoint_pairs", lib and ref_rounded)
    got = np.stack([np.asarray(D.decode_alpha_block(blk), np.int64).reshape(16) for blk in blocks])
    assert T.same(got, want), "" if isinstance(want, str) else int((want != got).sum())
