"""Hand-derived known-answer vectors (SURVEY.md section 4): they pin byte order, index remaps and the
degenerate paths independently of any implementation."""
import numpy as np
import pytest

import itw_testlib as T

CPU_APIS = ["oracle", "ref", "emu"]


def solid(v, a=255):
    img = np.full((4, 4, 4), v, np.uint8)
    img[..., 3] = a
    return img


@pytest.mark.parametrize("which", CPU_APIS)
def test_bc1_bc3_degenerate_blocks(which):
    api = getattr(T, which)()

    def check(fmt, v, want_hex, start=0):
        key = f"kat:{fmt}:solid{v}:{start}"
        if which == "ref":                         # the reference build, or what it produced where it is not built
            want = T.reference(key, api and (lambda: api.encode(fmt, solid(v))[start:]))
            assert T.same(np.frombuffer(bytes.fromhex(want_hex), np.uint8), want), key
        else:
            assert api.encode(fmt, solid(v))[start:].tobytes().hex() == want_hex, key
    # all-white: eps-only covariance, both endpoints 0xFFFF, NaN fast_quant -> indices 0 (quirk Q7)
    check("BC1", 255, "ffffffff00000000")
    check("BC1", 0, "0000000000000000")
    # mid grey: c0=127->0x7BEF, c1=128->0x8410, single-colour refine branch (K:424-432)
    check("BC1", 128, "1084108400000000")
    # BC3 alpha 255: ep1 = ep0+0.1, q = 0 -> 7 -> 8 -> 1 (K:557-560)
    check("BC3", 255, "ffff499224499224" + "ffffffff00000000")
    check("BC3", 128, "1084108400000000", start=8)


@pytest.mark.parametrize("which", CPU_APIS)
def test_bc4_bc5_endpoints_of_simple_blocks(which):
    api = getattr(T, which)()
    if api is None or which == "ref":
        pytest.skip("BC4/BC5 are not part of the ISPC reference build")
    # one texel 255, the rest 0: the 6-step fit finds no value strictly inside (0,1), leaves
    # (lo,hi) = (1,0) and breaks out at once (BC.h:783-789), so red_0 = 255 > red_1 = 0 and the
    # block decodes in 8-interpolant mode: texel 0 -> index 0, the zeros -> index 1.
    img = solid(0)
    img[0, 0, 0] = 255
    out = api.encode("BC4", img)
    assert (out[0], out[1]) == (255, 0)
    idx = int.from_bytes(out[2:8].tobytes(), "little")
    assert idx & 7 == 0 and all(((idx >> (3 * k)) & 7) == 1 for k in range(1, 16))
    # values {0,100,200}: touches 0 -> 6-interpolant mode, red_0 <= red_1, zeros take the explicit code 6
    img = solid(0)
    img[0, :, 0] = 100
    img[1, :, 0] = 200
    out = api.encode("BC4", img)
    assert out[0] <= out[1]
    idx = int.from_bytes(out[2:8].tobytes(), "little")
    assert all(((idx >> (3 * k)) & 7) == 6 for k in range(8, 16))
    # BC5 = two independent BC4 blocks of R and G
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (8, 8, 4), dtype=np.uint8)
    bc5 = api.encode("BC5", img).reshape(-1, 16)
    r = api.encode("BC4", img).reshape(-1, 8)
    g_img = img.copy()
    g_img[..., 0] = img[..., 1]
    g = api.encode("BC4", g_img).reshape(-1, 8)
    assert np.array_equal(bc5[:, :8], r) and np.array_equal(bc5[:, 8:], g)
