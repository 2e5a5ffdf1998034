"""The ABI takes arbitrary settings structs, not only the GetProfile_* presets.  Seeded random settings x random
blocks: the oracle must match the reference-source build, and the kernels (emulated on CPU, real on GPU) the oracle."""
import numpy as np
import pytest

import itw_testlib as T

B = T.binding


def random_bc7_settings(rng):
    s = B.Bc7Settings()
    for i in range(4):
        s.mode_selection[i] = bool(rng.integers(0, 2))
    if not any(s.mode_selection):
        s.mode_selection[int(rng.integers(0, 4))] = True
    for i in range(8):
        s.refineIterations[i] = int(rng.integers(0, 4))
    s.skip_mode2 = bool(rng.integers(0, 2))
    s.fastSkipTreshold_mode1 = int(rng.choice([0, 1, 3, 7, 20, 64]))
    s.fastSkipTreshold_mode3 = int(rng.choice([0, 1, 2, 9, 64]))
    s.channels = int(rng.choice([3, 4]))
    s.fastSkipTreshold_mode7 = int(rng.choice([0, 2, 5, 64])) if s.channels == 4 else 0
    s.mode45_channel0 = int(rng.integers(0, s.channels + 1))
    s.refineIterations_channel = int(rng.integers(0, 4))
    return s


def random_bc6_settings(rng):
    s = B.Bc6hSettings()
    s.slow_mode = bool(rng.integers(0, 2))
    s.fast_mode = bool(rng.integers(0, 2))
    s.refineIterations_1p = int(rng.integers(0, 4))
    s.refineIterations_2p = int(rng.integers(0, 4))
    s.fastSkipTreshold = int(rng.choice([0, 1, 3, 8, 17, 32]))
    return s


def images(rng, fmt):
    if fmt == "BC6H":
        a = rng.integers(0, 0x7C00, (8, 16, 4)).astype(np.uint16)
        b = (0x3400 + rng.integers(0, 300, (8, 16, 4))).astype(np.uint16)
        return [a, b]
    a = rng.integers(0, 256, (8, 16, 4), dtype=np.uint8)
    b = np.clip(100 + rng.normal(0, 25, (8, 16, 4)), 0, 255).astype(np.uint8)
    b[..., 3] = np.where(rng.random((8, 16)) < 0.3, 255, b[..., 3])
    return [a, b]


def copy_of(s):
    c = type(s)()
    import ctypes
    ctypes.memmove(ctypes.byref(c), ctypes.byref(s), ctypes.sizeof(s))
    return c


@pytest.mark.parametrize("seed", range(12))
def test_random_settings_cpu(seed):
    rng = np.random.default_rng(1000 + seed)
    ref = T.ref()
    for fmt, make in (("BC7", random_bc7_settings), ("BC6H", random_bc6_settings)):
        s = make(rng)
        for i, img in enumerate(images(rng, fmt)):
            want = T.oracle().encode(fmt, img, copy_of(s))
            ref_want = T.reference(f"random_settings:{seed}:{fmt}:{i}", ref and (lambda: ref.encode(fmt, img, copy_of(s))))
            assert T.same(want, ref_want), (fmt, seed, "oracle != reference build")
            assert np.array_equal(T.emu().encode(fmt, img, copy_of(s)), want), (fmt, seed, "emulated kernels != oracle")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(24))
def test_random_settings_gpu(seed):
    rng = np.random.default_rng(5000 + seed)
    lib = T.product()
    for fmt, make in (("BC7", random_bc7_settings), ("BC6H", random_bc6_settings)):
        s = make(rng)
        for img in images(rng, fmt):
            assert np.array_equal(lib.encode(fmt, img, copy_of(s)), T.oracle().encode(fmt, img, copy_of(s))), (fmt, seed)
