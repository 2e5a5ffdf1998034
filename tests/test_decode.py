"""Decoders (SURVEY.md 8f-3, include/itw_bcn.h section 5).

CPU: the kernels' per-block decode routines (csrc/decode.cuh, run through tests/emu) against the independent
numpy decoders of tests/bcn_decode.py -- on encoder output of every format/profile AND on random bit patterns
(every mode, reserved modes included).  GPU: itw_decode through the C-ABI against both."""
import os

import numpy as np
import pytest

import bcn_decode as D
import itw_testlib as T

LAYOUTS = D.bc6_layouts(open(os.path.join(T.ROOT, "oracle", "itw_oracle.cpp")).read())
FMTS = ["BC1", "BC3", "BC4", "BC5", "BC6H", "BC7"]


def reference_decode(fmt, blocks, w, h):
    """bcn_decode.py, with the documented behaviour for reserved modes (BC7: transparent black, BC6H: opaque black)."""
    bpb = 8 if fmt in ("BC1", "BC4") else 16
    blk = np.frombuffer(bytes(blocks), np.uint8).reshape(-1, bpb)
    out = np.zeros((h, w, 4), np.uint16 if fmt == "BC6H" else np.uint8)
    for i, b in enumerate(blk):
        by, bx = divmod(i, w // 4)
        try:
            px, _ = D.decode_image(fmt, b.tobytes(), 4, 4, LAYOUTS)
            if fmt == "BC6H":
                px = np.concatenate([px, np.full((4, 4, 1), 0x3C00)], axis=2)
        except ValueError:
            px = np.zeros((4, 4, 4), np.int64)
            if fmt == "BC6H":
                px[..., 3] = 0x3C00
        out[by * 4:by * 4 + 4, bx * 4:bx * 4 + 4] = px
    return out


def random_blocks(fmt, n, seed):
    bpb = 8 if fmt in ("BC1", "BC4") else 16
    rng = np.random.default_rng(seed)
    blk = rng.integers(0, 256, (n, bpb), dtype=np.uint8)
    if fmt == "BC7":                           # spread over the modes (a random byte is mode 0 half of the time)
        for i in range(n):
            m = i % 9
            blk[i, 0] = 0 if m == 8 else ((int(blk[i, 0]) & (0xFF ^ ((1 << (m + 1)) - 1))) | (1 << m))
    if fmt == "BC6H":                          # all 32 five-bit fields, reserved ones included
        for i in range(n):
            blk[i, 0] = (blk[i, 0] & 0xE0) | (i % 32)
    return blk.reshape(-1)


def encoded_streams(fmt):
    o = T.oracle()
    corpus = T.corpus_for(fmt)
    profs = {"BC7": ["slow", "alpha_slow", "alpha_fast"], "BC6H": ["bc6h_slow", "bc6h_veryfast"]}.get(fmt, [None])
    for prof in profs:
        for name in ("gradient", "smooth", "random") if fmt != "BC6H" else ("smooth", "lowvar", "random"):
            yield f"{prof}-{name}", T.run(o, fmt, corpus[name], prof)


@pytest.mark.parametrize("fmt", FMTS)
def test_emu_decode_matches_independent_decoder_on_encoder_output(fmt):
    e = T.emu()
    for tag, blocks in encoded_streams(fmt):
        got = e.decode(fmt, blocks, 64, 64)
        assert np.array_equal(got, reference_decode(fmt, blocks, 64, 64)), tag


@pytest.mark.parametrize("fmt", FMTS)
def test_emu_decode_matches_independent_decoder_on_random_bits(fmt):
    e = T.emu()
    blocks = random_blocks(fmt, 16 * 18, seed=5)
    got = e.decode(fmt, blocks, 64, 72)
    assert np.array_equal(got, reference_decode(fmt, blocks, 64, 72))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_gpu_decode_matches_emulation_and_independent_decoder(fmt):
    p, e = T.product(), T.emu()
    for tag, blocks in encoded_streams(fmt):
        got = p.decode(fmt, blocks, 64, 64)
        assert np.array_equal(got, e.decode(fmt, blocks, 64, 64)), tag
    blocks = random_blocks(fmt, 64 * 36, seed=9)
    got = p.decode(fmt, blocks, 256, 144)
    assert np.array_equal(got, e.decode(fmt, blocks, 256, 144))
    small = random_blocks(fmt, 16 * 18, seed=5)
    assert np.array_equal(p.decode(fmt, small, 64, 72), reference_decode(fmt, small, 64, 72))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["BC1", "BC7", "BC6H"])
def test_gpu_decode_device_pointers_and_strides(fmt):
    """device blocks -> device surface with a padded, (un)aligned stride gives the same texels as the host path."""
    import torch
    p = T.product()
    w, h = 128, 64
    blocks = random_blocks(fmt, (w // 4) * (h // 4), seed=3)
    want = p.decode(fmt, blocks, w, h)
    texel = want.strides[1]
    d_blocks = torch.from_numpy(blocks.copy()).cuda()
    for pad in (0, 16, 4):
        stride = w * texel + pad
        d_img = torch.zeros(h * stride, dtype=torch.uint8, device="cuda")
        p.decode_raw(fmt, d_blocks.data_ptr(), d_img.data_ptr(), w, h, stride)
        got = d_img.cpu().numpy().reshape(h, stride)[:, :w * texel].copy().view(want.dtype).reshape(h, w, 4)
        assert np.array_equal(got, want), pad
        # host destination with the same stride
        h_img = np.zeros(h * stride, np.uint8)
        p.decode_raw(fmt, d_blocks.data_ptr(), h_img.ctypes.data, w, h, stride)
        assert np.array_equal(h_img.reshape(h, stride)[:, :w * texel].copy().view(want.dtype).reshape(h, w, 4), want), pad


@pytest.mark.gpu
def test_gpu_encode_decode_round_trip_full_size():
    """Size-independent property at BASELINE's 4096^2: decode(encode(x)) is close to x (PSNR floors for BC1/BC7,
    at most one grey level off for the BC4 ramp on a slowly varying channel)."""
    import torch
    p = T.product()
    n = 4096
    yy, xx = np.mgrid[0:n, 0:n]
    img = np.stack([(xx // 16) & 255, (yy // 16) & 255, ((xx + yy) // 32) & 255, np.full_like(xx, 255)], axis=2).astype(np.uint8)
    d_img = torch.from_numpy(img).cuda()
    for fmt, floor in (("BC1", 40.0), ("BC7", 45.0)):
        bpb = 8 if fmt == "BC1" else 16
        d_blocks = torch.empty((n // 4) * (n // 4) * bpb, dtype=torch.uint8, device="cuda")
        p.encode_raw(fmt, d_img.data_ptr(), n, n, n * 4, d_blocks.data_ptr(), p.profile("veryfast") if fmt == "BC7" else None)
        d_out = torch.empty_like(d_img)
        p.decode_raw(fmt, d_blocks.data_ptr(), d_out.data_ptr(), n, n, n * 4)
        diff = (d_out[..., :3].float() - d_img[..., :3].float())
        mse = float((diff * diff).mean())
        psnr = 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)
        assert psnr >= floor, (fmt, psnr)
    d_blocks = torch.empty((n // 4) * (n // 4) * 8, dtype=torch.uint8, device="cuda")
    p.encode_raw("BC4", d_img.data_ptr(), n, n, n * 4, d_blocks.data_ptr())
    d_a = torch.empty_like(d_img)
    p.decode_raw("BC4", d_blocks.data_ptr(), d_a.data_ptr(), n, n, n * 4)
    assert int((d_a[..., 0].int() - d_img[..., 0].int()).abs().max()) <= 1


def _ref_decoders():
    """DirectXTex's own BC1 / BC3 decoder bodies, or None where they are not built."""
    import ctypes
    lib = T.ref_frontend()
    if lib is None:
        return None
    for name in ("ref_decode_bc1", "ref_decode_bc3"):
        getattr(lib, name).restype = None
        getattr(lib, name).argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    return lib


def _rounded(floats):
    """the UNORM8 store assumed for the preview: x * 255 + 0.5 truncated, evaluated in float32"""
    f = floats.astype(np.float32)
    return (f * np.float32(255.0) + np.float32(0.5)).astype(np.int64)


def test_bc1_bc3_decode_equals_directxtex_decoder_bodies_rounded():
    """csrc/decode.cuh (through the emulation) against DirectXTex's OWN DecodeBC1 / D3DXDecodeBC3 bodies (float texels,
    cut by oracle/build_ref_frontend.py), rounded to nearest: every 5- and 6-bit endpoint pair in both palette modes,
    every alpha endpoint pair, plus random blocks."""
    lib, e = _ref_decoders(), T.emu()
    blocks = []
    idx = 0
    for k in range(16):
        idx |= (k % 4) << (2 * k)
    idx_bytes = np.frombuffer(int(idx).to_bytes(4, "little"), np.uint8)
    for n0 in range(64):                                   # all endpoint pairs per channel (5-bit values repeat mod 32)
        for n1 in range(64):
            c0 = ((n0 & 31) << 11) | (n0 << 5) | (n1 & 31)
            c1 = ((n1 & 31) << 11) | (n1 << 5) | (n0 & 31)
            blocks.append(np.concatenate([np.frombuffer(int(c0).to_bytes(2, "little") + int(c1).to_bytes(2, "little"), np.uint8), idx_bytes]))
    rng = np.random.default_rng(12)
    blocks += [rng.integers(0, 256, 8, dtype=np.uint8) for _ in range(4096 - len(blocks) % 4096)]
    bc1 = np.concatenate(blocks)
    n = bc1.size // 8
    h = 4 * (n // 64)
    got = e.decode("BC1", bc1[: (h // 4) * 64 * 8], 256, h).reshape(h // 4, 4, 64, 4, 4).transpose(0, 2, 1, 3, 4).reshape(-1, 16, 4)
    want = T.reference("bc1_decode_rounded", lib and (lambda: _ref_decode_rounded(lib.ref_decode_bc1, bc1, 8, got.shape[0])))
    assert T.same(got.astype(np.int64), want), _first_differing(got, want)
    # BC3: colour block always in four-colour mode + every alpha endpoint pair
    blocks = []
    aidx = 0
    for k in range(16):
        aidx |= (k % 8) << (3 * k)
    aidx_bytes = np.frombuffer(int(aidx).to_bytes(6, "little"), np.uint8)
    for a0 in range(256):
        for a1 in range(0, 256, 3):
            colour = rng.integers(0, 256, 8, dtype=np.uint8)
            blocks.append(np.concatenate([np.array([a0, a1], np.uint8), aidx_bytes, colour]))
    blocks = blocks[: (len(blocks) // 64) * 64]
    bc3 = np.concatenate(blocks)
    h = 4 * (len(blocks) // 64)
    got = e.decode("BC3", bc3, 256, h).reshape(h // 4, 4, 64, 4, 4).transpose(0, 2, 1, 3, 4).reshape(-1, 16, 4)
    want = T.reference("bc3_decode_rounded", lib and (lambda: _ref_decode_rounded(lib.ref_decode_bc3, bc3, 16, got.shape[0])))
    assert T.same(got.astype(np.int64), want), _first_differing(got, want)


def _ref_decode_rounded(fn, blocks, bpb, n):
    """n blocks of `bpb` bytes through a DirectXTex decoder body, rounded like the preview store: (n, 16, 4) int64"""
    out = np.zeros((n, 64), np.float32)
    for i in range(n):
        blk = np.ascontiguousarray(blocks[bpb * i:bpb * i + bpb])
        fn(blk.ctypes.data, out[i].ctypes.data)
    return _rounded(out).reshape(n, 16, 4)


def _first_differing(got, want):
    if isinstance(want, str):
        return "differs from the stored digest of DirectXTex's decode"
    return int(np.nonzero((got.astype(np.int64) != want).any(axis=(1, 2)))[0][0])
