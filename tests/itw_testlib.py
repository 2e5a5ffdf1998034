"""Shared helpers of the test-suite: library loaders and the input corpus.

oracle(), ref() and emu() load TEST INFRASTRUCTURE (oracle/, tests/emu); product() loads the
library under test.  Nothing here reads the reference checkout; reference() and same() let a test compare with the
reference's own code where oracle/_ref is built and with the digests that code left in tests/golden elsewhere."""
import atexit
import functools
import hashlib
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
pkg = importlib.import_module("intel-texture-works-plugin_b200")
binding = importlib.import_module("intel-texture-works-plugin_b200.binding")
synth = pkg.synth

ORACLE_SO = os.path.join(ROOT, "oracle", "libitw_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libitw_ref.so")
EMU_SO = os.path.join(ROOT, "tests", "emu", "libitw_emu.so")


@functools.lru_cache(None)
def oracle():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    return binding.EncoderApi(ORACLE_SO, "oracle_")


@functools.lru_cache(None)
def ref():
    """The reference's own sources compiled scalar (oracle/build_ref.py); None if unavailable."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import build_ref
        try:
            build_ref.build(verbose=False)
        except FileNotFoundError:
            return None
    finally:
        sys.path.pop(0)
    return binding.EncoderApi(REF_SO, "")


@functools.lru_cache(None)
def ref_frontend():
    """The reference's own front-end function bodies (oracle/build_ref_frontend.py) as a ctypes library; None if unavailable."""
    import ctypes
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import build_ref_frontend
        try:
            path = build_ref_frontend.build(verbose=False)
        except FileNotFoundError:
            return None
    finally:
        sys.path.pop(0)
    lib = ctypes.CDLL(path)
    lib.ref_convert_pixels.restype = ctypes.c_int
    lib.ref_convert_pixels.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_uint, ctypes.c_void_p]
    lib.ref_mip_chain_f16.restype = ctypes.c_int
    lib.ref_mip_chain_f16.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.ref_float_to_half.restype = ctypes.c_ushort
    lib.ref_float_to_half.argtypes = [ctypes.c_float]
    lib.ref_half_to_float.restype = ctypes.c_float
    lib.ref_half_to_float.argtypes = [ctypes.c_ushort]
    return lib


# ---------------------------------------------------------------------------------------------
# results of the reference's own code: live from oracle/_ref where it is built, else the stored digests
# ---------------------------------------------------------------------------------------------
REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")
_RECORD = os.environ.get("ITW_RECORD_REFERENCE")       # set by tests/golden/make_golden_reference.py
_recorded = {}


def digest(a):
    """dtype, shape and the first 128 bits of the SHA-256 of an array's bytes; -0.0 and 0.0 hash alike, as they compare equal."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)
    return f"{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()[:32]}"


@functools.lru_cache(None)
def _stored():
    with open(REF_DIGESTS) as f:
        return json.load(f)["digests"]


def _write_recorded():
    out = {"generator": "tests/golden/make_golden_reference.py", "digests": {}}
    if os.path.exists(_RECORD):
        with open(_RECORD) as f:
            out = json.load(f)
    out["digests"].update(_recorded)
    out["digests"] = dict(sorted(out["digests"].items()))
    with open(_RECORD, "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")


def reference(key, live):
    """What the reference's own code computes for `key`.  `live` computes it (an array) where the reference build is
    available and is None elsewhere.  Returns the array when computed live (after checking it against the stored digest,
    so that the golden file cannot drift from the reference), else the digest stored in tests/golden/reference_digests.json.
    Compare the result with same()."""
    if _RECORD:
        assert live is not None, f"{key}: recording needs the reference build"
        want = np.ascontiguousarray(live())
        d = digest(want)
        assert _recorded.setdefault(key, d) == d, f"{key}: two different results under one key"
        if len(_recorded) == 1:
            atexit.register(_write_recorded)
        return want
    stored = _stored().get(key)
    assert stored is not None, f"{key}: no stored reference digest (run tests/golden/make_golden_reference.py)"
    if live is None:
        return stored
    want = np.ascontiguousarray(live())
    assert digest(want) == stored, f"{key}: the reference build no longer gives the stored result"
    return want


def same(got, want):
    """got equals a result of reference() in dtype, shape and every element.  Live or stored, the comparison is the same
    one (by digest), so a test passes with the reference build exactly when it passes without."""
    return digest(got) == (want if isinstance(want, str) else digest(want))


@functools.lru_cache(None)
def emu():
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    try:
        import build_emu
        build_emu.build(verbose=False)
    finally:
        sys.path.pop(0)
    return binding.EncoderApi(EMU_SO, "emu_")


@functools.lru_cache(None)
def product():
    return pkg.ItwBcn()


# ---------------------------------------------------------------------------------------------
# corpus: small images that reach every code path (all BC7 modes, all BC6H modes, degenerate blocks)
# ---------------------------------------------------------------------------------------------
def corpus8(size=64, seed=7):
    rng = np.random.default_rng(seed)
    n = size
    out = {}
    out["random"] = synth.random_rgba8(n, n, seed=seed)
    out["gradient"] = synth.gradient_rgba8(n, n)
    lv = (rng.integers(0, 4, (n, n, 4)) * 64 + rng.integers(0, 8, (n, n, 4))).astype(np.uint8)
    out["lowvar"] = lv
    out["flat"] = np.repeat(np.repeat(rng.integers(0, 256, (n // 4, n // 4, 4), dtype=np.uint8), 4, 0), 4, 1)
    a = rng.integers(0, 256, (n, n, 4), dtype=np.uint8)
    a[..., 3] = np.where(rng.random((n, n)) < 0.5, 255, 0)
    out["alpha01"] = a
    s = rng.integers(0, 256, (n, n, 4), dtype=np.uint8)
    s[..., :3] = np.clip(128 + rng.normal(0, 10, (n, n, 3)), 0, 255).astype(np.uint8)
    out["smooth"] = s
    two = np.zeros((n, n, 4), np.uint8)
    pick = rng.random((n, n)) < 0.5
    two[pick] = (250, 10, 30, 255)
    two[~pick] = (20, 200, 90, 128)
    out["twocolour"] = two
    edge = np.zeros((n, n, 4), np.uint8)
    edge[..., 3] = 255
    edge[:, : n // 2, :3] = 255
    edge[5::9, 3::7, :3] = 0                       # single outliers
    out["extremes"] = edge
    out["mixed"] = synth.mixed_rgba8(n, n)
    return out


def corpus16(size=64, seed=11):
    rng = np.random.default_rng(seed)
    n = size
    out = {}
    out["random"] = synth.random_rgba16f(n, n, seed=seed)
    out["signbits"] = rng.integers(0, 65536, (n, n, 4)).astype(np.uint16)       # quirk Q10
    x = np.arange(n, dtype=np.float32)
    v = np.exp2((x[None, :] + x[:, None]) / 16 - 4)
    out["smooth"] = np.stack([v * (1 + c / 8) for c in range(4)], -1).astype(np.float16).view(np.uint16)
    out["flat"] = np.repeat(np.repeat(rng.integers(0, 0x7C00, (n // 4, n // 4, 4)), 4, 0), 4, 1).astype(np.uint16)
    out["lowvar"] = rng.integers(0x3000, 0x3100, (n, n, 4)).astype(np.uint16)
    out["zeros"] = np.zeros((n, n, 4), np.uint16)
    out["maxhalf"] = np.full((n, n, 4), 0x7BFF, np.uint16)
    nar = (0x3800 + rng.integers(0, 40, (n, n, 4))).astype(np.uint16)          # tiny spans -> modes 2-4, 13
    nar[..., 0] += rng.integers(0, 200, (n, n)).astype(np.uint16)
    out["narrow"] = nar
    for c, tag in ((1, "narrow_g"), (2, "narrow_b")):                          # wide channel G / B -> modes 3,7 / 4,8
        v = (0x3800 + rng.integers(0, 40, (n, n, 4))).astype(np.uint16)
        v[..., c] += rng.integers(0, 200, (n, n)).astype(np.uint16)
        v[: n // 2, :, c] += rng.integers(0, 1500, (n // 2, n)).astype(np.uint16)
        out[tag] = v
    return out


ALL_CASES = ([("BC1", None), ("BC3", None), ("BC4", None), ("BC5", None)]
             + [("BC7", p) for p in binding.BC7_PROFILES] + [("BC6H", p) for p in binding.BC6H_PROFILES])


def corpus_for(fmt, size=64):
    return corpus16(size) if fmt == "BC6H" else corpus8(size)


def run(api, fmt, img, prof):
    return api.encode(fmt, img, api.profile(prof) if prof else None)


def differing_blocks(a, b, bpb):
    return int((a.reshape(-1, bpb) != b.reshape(-1, bpb)).any(1).sum())


def oracle_mip_chain_rgba8(img, srgb=0, levels=None, pad=True):
    """The RGBA8 mip chain contract (include/itw_bcn.h section 4): DirectXTex's non-WIC generators as restated in
    oracle/itw_oracle_frontend.cpp (oracle_mip_chain_rgba8; pinned to the reference's own bodies by tests/test_mips.py).
    Returns the list of levels, each padded to multiples of 4 by edge replication unless pad=False."""
    import ctypes
    h, w = img.shape[:2]
    if levels is None:
        levels = max(h, w).bit_length()
    dims = [(max(1, h >> l), max(1, w >> l)) for l in range(levels)]
    out = np.zeros(sum(a * b * 4 for a, b in dims), np.uint8)
    src = np.ascontiguousarray(img)
    f = oracle().lib.oracle_mip_chain_rgba8
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    assert f(src.ctypes.data, w, h, levels, int(srgb), out.ctypes.data) == 0
    res, off = [], 0
    for a, b in dims:
        lvl = out[off:off + a * b * 4].reshape(a, b, 4)
        res.append(synth.pad_to_4(lvl) if pad else lvl)
        off += a * b * 4
    return res
