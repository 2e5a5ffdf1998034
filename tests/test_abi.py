"""C-ABI checks that need no GPU: struct layouts, exported symbols, profile tables."""
import ctypes
import os
import re

import numpy as np
import pytest

import itw_testlib as T

B = T.binding


def test_struct_layouts():
    # ispc_texcomp.h:19-50 on LP64
    assert ctypes.sizeof(B.RgbaSurface) == 24
    assert (B.RgbaSurface.width.offset, B.RgbaSurface.height.offset, B.RgbaSurface.stride.offset) == (8, 12, 16)
    assert ctypes.sizeof(B.Bc7Settings) == 64
    assert B.Bc7Settings.refineIterations.offset == 4
    assert B.Bc7Settings.skip_mode2.offset == 36
    assert B.Bc7Settings.fastSkipTreshold_mode1.offset == 40
    assert B.Bc7Settings.channels.offset == 60
    assert ctypes.sizeof(B.Bc6hSettings) == 16
    assert (B.Bc6hSettings.fast_mode.offset, B.Bc6hSettings.refineIterations_1p.offset,
            B.Bc6hSettings.fastSkipTreshold.offset) == (1, 4, 12)


def test_library_loads_and_exports_every_declared_symbol():
    lib = T.product()          # loads libitw_bcn.so; no CUDA call is made
    header = open(os.path.join(T.ROOT, "include", "itw_bcn.h")).read()
    declared = set(re.findall(r"\b((?:GetProfile_|CompressBlocks|CompressImage|itw_)\w+|GetProcessorCount|InitWin32Threads|DestroyThreads|GetBytesPerBlock)\s*\(", header))
    assert declared == set(B.EXPORTS), declared ^ set(B.EXPORTS)
    for name in declared:
        assert getattr(lib.lib, name) is not None, name
    assert lib.lib.itw_bytes_per_block(71) == 8 and lib.lib.itw_bytes_per_block(98) == 16
    assert lib.lib.itw_bytes_per_block(95) == 16 and lib.lib.itw_bytes_per_block(1) == 0
    assert lib.last_error() == ""


def _fields(s):
    out = {}
    for name, _ in s._fields_:
        v = getattr(s, name)
        out[name] = list(v) if hasattr(v, "__len__") else v
    return out


# known answers: 3rdParty/Intel/Source/ispc_texcomp.cpp:20-410, field by field
BC7_KAT = {
    "ultrafast": dict(channels=3, sel=[0, 0, 0, 1], skip2=1, t=(3, 1, 0), refine=[2, 2, 2, 1, 2, 2, 1], ch0=0, rch=0),
    "veryfast": dict(channels=3, sel=[0, 1, 0, 1], skip2=1, t=(3, 1, 0), refine=[2, 2, 2, 1, 2, 2, 1], ch0=0, rch=0),
    "fast": dict(channels=3, sel=[0, 1, 0, 1], skip2=1, t=(12, 4, 0), refine=[2, 2, 2, 1, 2, 2, 2], ch0=0, rch=0),
    "basic": dict(channels=3, sel=[1, 1, 1, 1], skip2=1, t=(12, 8, 0), refine=[2, 2, 2, 2, 2, 2, 2], ch0=0, rch=2),
    "slow": dict(channels=3, sel=[1, 1, 1, 1], skip2=0, t=(64, 64, 0), refine=[4, 4, 4, 4, 4, 4, 4], ch0=0, rch=4),
    "alpha_ultrafast": dict(channels=4, sel=[0, 0, 1, 1], skip2=1, t=(0, 0, 4), refine=[2, 1, 2, 1, 1, 1, 2, 2], ch0=3, rch=1),
    "alpha_veryfast": dict(channels=4, sel=[0, 1, 1, 1], skip2=1, t=(0, 0, 4), refine=[2, 1, 2, 1, 2, 2, 2, 2], ch0=3, rch=2),
    "alpha_fast": dict(channels=4, sel=[0, 1, 1, 1], skip2=1, t=(4, 4, 8), refine=[2, 1, 2, 1, 2, 2, 2, 2], ch0=3, rch=2),
    "alpha_basic": dict(channels=4, sel=[1, 1, 1, 1], skip2=1, t=(12, 8, 8), refine=[2, 2, 2, 2, 2, 2, 2, 2], ch0=0, rch=2),
    "alpha_slow": dict(channels=4, sel=[1, 1, 1, 1], skip2=0, t=(64, 64, 64), refine=[4, 4, 4, 4, 4, 4, 4, 4], ch0=0, rch=4),
}
BC6_KAT = {"bc6h_veryfast": (0, 1, 0, 0, 0), "bc6h_fast": (0, 1, 2, 0, 1), "bc6h_basic": (0, 0, 4, 2, 2),
           "bc6h_slow": (1, 0, 10, 2, 2), "bc6h_veryslow": (1, 0, 32, 2, 2)}


def _profile_bytes(api, name):
    return np.frombuffer(bytes(api.profile(name)), np.uint8)


def _reference_profile(name):
    """The reference build's GetProfile_<name>: its struct bytes live, their stored digest elsewhere."""
    ref = T.ref()
    return T.reference(f"profile:{name}", ref and (lambda: _profile_bytes(ref, name)))


class _ProfilesEqualToReference:
    """Where the reference build is not available: the product's profiles, each checked byte for byte against the
    reference's stored result, so that the known answers below are asserted on the reference's values."""

    def profile(self, name):
        assert T.same(_profile_bytes(T.product(), name), _reference_profile(name)), name
        return T.product().profile(name)


@pytest.mark.parametrize("which", ["product", "oracle", "ref"])
def test_profiles_known_answers(which):
    api = getattr(T, which)()
    if api is None:
        api = _ProfilesEqualToReference()
    for name, k in BC7_KAT.items():
        s = api.profile(name)
        assert s.channels == k["channels"], name
        assert [int(x) for x in s.mode_selection] == k["sel"], name
        assert int(s.skip_mode2) == k["skip2"], name
        assert (s.fastSkipTreshold_mode1, s.fastSkipTreshold_mode3, s.fastSkipTreshold_mode7) == k["t"], name
        n = len(k["refine"])
        assert list(s.refineIterations)[:n] == k["refine"], name
        if n == 7:
            assert s.refineIterations[7] == 0, "RGB profiles leave refineIterations[7] untouched"
        assert (s.mode45_channel0, s.refineIterations_channel) == (k["ch0"], k["rch"]), name
    for name, k in BC6_KAT.items():
        s = api.profile(name)
        assert (int(s.slow_mode), int(s.fast_mode), s.fastSkipTreshold, s.refineIterations_1p, s.refineIterations_2p) == k


def test_profiles_identical_across_implementations():
    apis = [a for a in (T.product(), T.oracle(), T.ref()) if a is not None]
    for name in B.BC7_PROFILES + B.BC6H_PROFILES:
        got = [_fields(a.profile(name)) for a in apis]
        assert all(g == got[0] for g in got), name
        assert T.same(_profile_bytes(T.product(), name), _reference_profile(name)), name


def test_no_cpu_fallback_when_there_is_no_gpu():
    """On a machine without a CUDA device every compute entry point must FAIL LOUDLY (error string, output untouched):
    the product has no CPU path.  (Skipped where a GPU exists.)"""
    import ctypes
    import numpy as np
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a CUDA device is present")
    except ImportError:
        pass
    lib = T.product()
    img = np.full((8, 8, 4), 77, np.uint8)
    out = np.full(4 * 16, 0xAB, np.uint8)
    surf = T.binding.RgbaSurface(img.ctypes.data, 8, 8, 32)
    for fmt, settings in (("BC1", None), ("BC3", None), ("BC4", None), ("BC5", None), ("BC7", lib.profile("veryfast"))):
        out[:] = 0xAB
        with pytest.raises(RuntimeError, match="libitw_bcn"):
            lib.encode_raw(fmt, img.ctypes.data, 8, 8, 32, out.ctypes.data, settings)
        assert (out == 0xAB).all(), fmt                      # nothing was written
    with pytest.raises(RuntimeError):
        lib.decode("BC1", np.zeros(32, np.uint8), 8, 8)
    with pytest.raises(RuntimeError):
        lib.convert_pixels("BC7", img, 1)
    assert lib.last_error() != ""
