"""The GPU encoders on real, alpha and degenerate content, at every profile and every launch shape.

Content: the reference's sample images (tests/golden/sample_images.npz, including monkey.png's real 0..255 alpha, a normal map
and a smooth grey ramp), the test corpus, and a deterministic catalogue of degenerate blocks made below (flat blocks at every
value, two colours one LSB or far apart, lone outliers, alpha-only variation, 0/255-only blocks; for HDR every pair of the
special halves -- zeros, denormals, the largest finite values, infinities, NaNs, negatives -- plus near-flat blocks).

Every BCn block is encoded from its own sixteen texels alone, so these sources are gathered into one POOL of unique blocks per
pixel format.  The oracle's encoding of the pool, one result per block and profile, is pinned to the reference's own code
(live from oracle/_ref where it is built, from tests/golden/reference_digests.json elsewhere), and so is every image's and the
catalogue's encoding, which is that result gathered by the image's block indices.  The GPU tests then encode

* each sample image whole, against the stored reference digests, and
* MOSAICS: surfaces of up to ~61 k blocks made of a seeded permutation of the pool, sized from the SM count so that they reach
  the launch switches (eight- and sixteen-block BC7 rounds, several rounds per CTA, both BC6H stage buffers, ragged tails),
  through every entry point; the expectation is the oracle's pool result gathered by the same permutation.

A mismatch is reported per block: mosaic coordinate, source (image and block position, or catalogue family) and the expected
and actual BC7 / BC6H mode."""
import ctypes
import functools
import os
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import itw_testlib as T
import test_bc45_vs_directxtex as BX

SAMPLES = os.path.join(os.path.dirname(__file__), "golden", "sample_images.npz")
LDR_SAMPLES = ("baboon.png", "gradients.png", "colors-260K.png", "colors-16M.png", "juggling-balls.jpg", "monkey.png", "normals.png",
               "radial-grayscale.png")
HDR_SAMPLES = ("HDR.hdr", "monkey-32bit.hdr")
NEW_SAMPLES = ("monkey.png", "normals.png", "radial-grayscale.png", "monkey-32bit.hdr")
BC45 = ("BC4", "BC5")


@functools.lru_cache(None)
def sample(name):
    with np.load(SAMPLES) as z:
        return np.ascontiguousarray(z[name])


# ---------------------------------------------------------------------------------------------
# the degenerate-block catalogue: family -> (n, 16, 4) blocks, row-major texels
# ---------------------------------------------------------------------------------------------
def _flat(colours):
    return np.repeat(np.asarray(colours)[:, None, :], 16, 1)


def _two(c1, c2, mask):
    return np.where(mask[..., None], c1[:, None, :], c2[:, None, :])


@functools.lru_cache(None)
def ldr_catalogue():
    rng = np.random.default_rng(2024)
    v = np.arange(256)
    opaque = np.full(256, 255)
    zero = np.zeros(256, int)
    fam = {}
    # flat blocks at every value: grey, each channel alone, and a mixed colour (alpha varies too)
    fam["flat-grey"] = _flat(np.stack([v, v, v, opaque], 1))
    for c, tag in enumerate("rgb"):
        fam[f"flat-{tag}"] = _flat(np.stack([v if k == c else zero for k in range(3)] + [opaque], 1))
    fam["flat-alpha"] = _flat(np.stack([zero, zero, zero, v], 1))
    fam["flat-mixed"] = _flat(np.stack([v, 255 - v, (v * 37 + 11) % 256, (v * 101 + 7) % 256], 1))
    # two colours one LSB apart in one channel (coincident endpoints after quantisation), under random masks; half opaque
    c1 = rng.integers(0, 256, (256, 4))
    c1[:128, 3] = 255
    c2 = c1.copy()
    k = rng.integers(0, 4, 256)
    c2[np.arange(256), k] += np.where(c1[np.arange(256), k] < 255, 1, -1)
    fam["two-close"] = _two(c1, c2, rng.random((256, 16)) < 0.5)
    # two colours far apart under random masks (one texel of one colour included); half opaque
    c1 = rng.integers(0, 256, (256, 4))
    c2 = 255 - c1 // 4
    c1[:128, 3] = c2[:128, 3] = 255
    m = rng.random((256, 16)) < rng.random((256, 1))
    m[:32] = False
    m[np.arange(32), rng.integers(0, 16, 32)] = True
    fam["two-far"] = _two(c1, c2, m)
    # a flat block with one outlier texel
    base = rng.integers(0, 256, (128, 4))
    base[:64, 3] = 255
    blk = _flat(base).copy()
    blk[np.arange(128), rng.integers(0, 16, 128)] = rng.integers(0, 256, (128, 4))
    fam["outlier"] = blk
    # flat colour with varying alpha, and with alpha 0 / 255 only
    blk = _flat(rng.integers(0, 256, (64, 4))).copy()
    blk[..., 3] = rng.integers(0, 256, (64, 16))
    fam["alpha-varying"] = blk
    blk = _flat(rng.integers(0, 256, (64, 4))).copy()
    blk[..., 3] = np.where(rng.random((64, 16)) < 0.5, 0, 255)
    fam["alpha-0-255"] = blk
    # blocks made only of 0 and 255, per channel and per texel
    fam["extremes"] = np.where(rng.random((128, 16, 4)) < 0.5, 0, 255)
    fam["black-white"] = np.repeat(np.where(rng.random((64, 16, 1)) < 0.5, 0, 255), 4, 2)
    return {f: np.ascontiguousarray(b.astype(np.uint8)) for f, b in fam.items()}


HALVES = (0x0000, 0x0001, 0x0002, 0x03FF, 0x0400, 0x3BFF, 0x3C00, 0x7BFE, 0x7BFF, 0x7C00, 0x7C01, 0x7E00, 0x7FFF, 0x8000, 0x8001,
          0xBC00, 0xFBFF, 0xFC00, 0xFFFF)


@functools.lru_cache(None)
def hdr_catalogue():
    rng = np.random.default_rng(2025)
    h = np.array(HALVES)
    a, b = np.repeat(h, len(h)), np.tile(h, len(h))                  # every ordered pair
    one = np.full(a.size, 0x3C00)
    fam = {}
    fam["hdr-flat-pair"] = _flat(np.stack([a, b, a, one], 1))
    ca, cb = np.stack([a, a, a, one], 1), np.stack([b, b, b, one], 1)
    fam["hdr-two-valued"] = _two(ca, cb, rng.random((a.size, 16)) < 0.5)
    fam["hdr-channel-mix"] = np.where(rng.random((a.size, 16, 4)) < 0.5, ca[:, None, :], cb[:, None, :])
    base = np.repeat(h, 8)
    noisy = (base[:, None, None] + rng.integers(-2, 3, (base.size, 16, 4))) & 0xFFFF      # +-2 ulp around each special half
    noisy[..., 3] = 0x3C00
    fam["hdr-near-flat"] = noisy
    return {f: np.ascontiguousarray(x.astype(np.uint16)) for f, x in fam.items()}


# ---------------------------------------------------------------------------------------------
# blocks <-> surfaces
# ---------------------------------------------------------------------------------------------
def blocks_of(img):
    h, w, c = img.shape
    return img.reshape(h // 4, 4, w // 4, 4, c).transpose(0, 2, 1, 3, 4).reshape(-1, 16, c)


def surface_of(blocks, width):
    """Blocks laid out row-major on a surface `width` blocks wide (the last row completed with copies of block 0)."""
    n = len(blocks)
    rows = -(-n // width)
    if rows * width > n:
        blocks = np.concatenate([blocks, np.repeat(blocks[:1], rows * width - n, 0)])
    c = blocks.shape[2]
    return np.ascontiguousarray(blocks.reshape(rows, width, 4, 4, c).transpose(0, 2, 1, 3, 4).reshape(4 * rows, 4 * width, c))


def encode_blocks(api, fmt, prof, blocks, width=64):
    """Encode each block with `api` (one result row per block), four-texel-row strips in parallel."""
    img = surface_of(blocks, width)
    settings = api.profile(prof) if prof else None
    strips = [np.ascontiguousarray(img[y:y + 4]) for y in range(0, img.shape[0], 4)]
    with ThreadPoolExecutor(min(8, os.cpu_count() or 1)) as ex:
        out = list(ex.map(lambda s: api.encode(fmt, s, settings), strips))
    return np.concatenate(out).reshape(-1, T.binding.FORMATS[fmt][1])[:len(blocks)]


# ---------------------------------------------------------------------------------------------
# the pool: unique blocks of corpus + sample images + catalogue, in order of first appearance
# ---------------------------------------------------------------------------------------------
class Pool:
    def __init__(self, sources):
        """sources: list of (name, blocks, width in blocks or None for a catalogue family)."""
        self.sources = sources
        allb = np.concatenate([b for _, b, _ in sources])
        flat = np.ascontiguousarray(allb.reshape(len(allb), -1))
        _, first, inverse = np.unique(flat.view(np.dtype((np.void, flat.shape[1] * flat.itemsize))).ravel(),
                                      return_index=True, return_inverse=True)
        order = np.argsort(first)
        rank = np.empty_like(order)
        rank[order] = np.arange(len(order))
        self.first = first[order]                           # index into the concatenated sources of each pool block
        self.blocks = np.ascontiguousarray(allb[self.first])
        where = rank[inverse.ravel()]                       # pool index of every source block
        self.index, self._starts, off = {}, [], 0
        for name, b, _ in sources:
            self.index[name] = where[off:off + len(b)]
            self._starts.append(off)
            off += len(b)

    def __len__(self):
        return len(self.blocks)

    def origin(self, i):
        """Where pool block i first appears: image name and block position, or catalogue family and number."""
        g = int(self.first[i])
        k = int(np.searchsorted(self._starts, g, side="right")) - 1
        name, _, width = self.sources[k]
        j = g - self._starts[k]
        return f"{name} block ({j % width}, {j // width})" if width else f"catalogue {name} #{j}"

    def catalogue_index(self):
        return np.concatenate([self.index[n] for n, _, w in self.sources if w is None])


@functools.lru_cache(None)
def pool(hdr):
    corpus = T.corpus16() if hdr else T.corpus8()
    srcs = [(f"corpus {n}", blocks_of(img), img.shape[1] // 4) for n, img in corpus.items()]
    srcs += [(n, blocks_of(sample(n)), sample(n).shape[1] // 4) for n in (HDR_SAMPLES if hdr else LDR_SAMPLES)]
    srcs += [(f, b, None) for f, b in (hdr_catalogue() if hdr else ldr_catalogue()).items()]
    return Pool(srcs)


def pool_for(fmt):
    return pool(fmt == "BC6H")


def pool_key(fmt, prof):
    return f"bc45:{fmt}:pool" if fmt in BC45 else f"pool:{fmt}:{prof}"


@functools.lru_cache(None)
def expectation(fmt, prof):
    """The oracle's result for every pool block (rows of bytes)."""
    return encode_blocks(T.oracle(), fmt, prof, pool_for(fmt).blocks)


@functools.lru_cache(None)
def _reference_pool_live(fmt, prof):
    blocks = pool_for(fmt).blocks
    if fmt in BC45:
        return BX.ref_encode(BX.ref_lib(), fmt, surface_of(blocks, len(blocks))).reshape(len(blocks), -1)
    return encode_blocks(T.ref(), fmt, prof, blocks)


def reference_live(fmt):
    """Whether the reference's own code for fmt is built here."""
    return (BX.ref_lib() if fmt in BC45 else T.ref()) is not None


def reference_gathered(key, fmt, prof, index):
    """The reference's result for the blocks `index` of the pool: live (the reference's pool result, gathered) or stored."""
    live = (lambda: _reference_pool_live(fmt, prof)[index].reshape(-1)) if reference_live(fmt) else None
    return T.reference(key, live)


# ---------------------------------------------------------------------------------------------
# modes and the mismatch report
# ---------------------------------------------------------------------------------------------
def bc7_mode(row):
    b = int(row[0])
    return (b & -b).bit_length() - 1 if b else None             # mode m starts with m zero bits and a one


def bc6h_mode(row):
    b = int(row[0])
    return b & 3 if (b & 3) < 2 else b & 31                     # 2-bit mode field for modes 1, 2; 5-bit field otherwise


def modes(fmt, rows):
    if fmt == "BC7":
        return np.array([-1 if r[0] == 0 else bc7_mode(r) for r in rows])          # -1: no valid mode
    return np.array([bc6h_mode(r) for r in rows])


def mismatch_report(got, want, fmt, idx, width, pl, limit=8):
    """'' when equal; else the number of differing blocks and, for the first `limit`, their mosaic coordinate, pool origin and
    expected / actual bytes (and mode for BC7 / BC6H)."""
    bpb = T.binding.FORMATS[fmt][1]
    got, want = np.asarray(got).reshape(-1, bpb), np.asarray(want).reshape(-1, bpb)
    bad = np.flatnonzero((got != want).any(1))
    if bad.size == 0:
        return ""
    mode = {"BC7": bc7_mode, "BC6H": bc6h_mode}.get(fmt)
    lines = [f"{fmt}: {bad.size} of {len(want)} blocks differ"]
    for b in bad[:limit]:
        m = f" mode {mode(want[b])} expected, {mode(got[b])} got;" if mode else ""
        lines.append(f"  mosaic block ({b % width}, {b // width}) = pool block {idx[b]} from {pl.origin(idx[b])}:{m}"
                     f" expected {want[b].tobytes().hex()}, got {got[b].tobytes().hex()}")
    return "\n".join(lines)


def mosaic(fmt, wb, hb, seed):
    """A wb x hb-block surface made of a seeded permutation of the pool (repeated as needed), and the pool index of each of
    its blocks (row-major)."""
    pl = pool_for(fmt)
    rng = np.random.default_rng(seed)
    n = wb * hb
    idx = np.concatenate([rng.permutation(len(pl)) for _ in range(-(-n // len(pl)))])[:n]
    return surface_of(pl.blocks[idx], wb), idx


# ---------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------
# modes each profile emits on the pool (BC7: mode number; BC6H: mode field), at least MODE_FLOOR blocks each
MODE_FLOOR = 3
BC6H_ALL = (0, 1, 2, 6, 10, 14, 18, 22, 26, 30, 3, 7, 11, 15)
EXPECTED_MODES = {
    "ultrafast": (6,), "veryfast": (1, 3, 6), "fast": (1, 3, 6), "basic": (0, 1, 3, 4, 5, 6), "slow": (0, 1, 2, 3, 4, 5, 6),
    "alpha_ultrafast": (4, 5, 6), "alpha_veryfast": (4, 5, 6, 7), "alpha_fast": (1, 3, 4, 5, 6, 7),
    "alpha_basic": (0, 1, 3, 4, 5, 6, 7), "alpha_slow": (0, 1, 2, 3, 4, 5, 6, 7),
    "bc6h_veryfast": (3, 7, 11, 15), "bc6h_fast": BC6H_ALL, "bc6h_basic": BC6H_ALL, "bc6h_slow": BC6H_ALL, "bc6h_veryslow": BC6H_ALL,
}
CASE_IDS = [f"{f}-{p}" for f, p in T.ALL_CASES]
MODE_CASES = [c for c in T.ALL_CASES if c[0] in ("BC7", "BC6H")]


def test_catalogue_reaches_the_edges():
    ldr, hdr = ldr_catalogue(), hdr_catalogue()
    assert sum(len(b) for b in ldr.values()) > 2000 and sum(len(b) for b in hdr.values()) > 1000
    grey = ldr["flat-grey"]
    assert np.array_equal(grey[:, 0, 0], np.arange(256)) and (grey == grey[:, :1]).all()
    tc = ldr["two-close"].astype(int)
    assert all(np.abs(b.max(0) - b.min(0)).sum() <= 1 for b in tc)
    for h in HALVES:
        assert (hdr["hdr-flat-pair"][..., 0] == h).all(1).any()
    assert (hdr["hdr-two-valued"] == 0x7E00).any() and (hdr["hdr-two-valued"] == 0xFC00).any()
    assert (ldr["alpha-0-255"][..., 3] == 0).any()
    alpha = sample("monkey.png")[..., 3]                               # real alpha: soft edges over the whole range
    assert alpha.min() == 0 and alpha.max() == 255 and len(np.unique(alpha)) > 250


@pytest.mark.parametrize("fmt,prof", T.ALL_CASES, ids=CASE_IDS)
def test_pool_oracle_equals_reference(fmt, prof):
    """Pool pin: the oracle's result on every unique block equals the reference's own code's (stored digest or live)."""
    want = T.reference(pool_key(fmt, prof), (lambda: _reference_pool_live(fmt, prof)) if reference_live(fmt) else None)
    got = expectation(fmt, prof)
    assert T.same(got, want), (fmt, prof) + (() if isinstance(want, str) else (T.differing_blocks(got, want, got.shape[1]),))


@pytest.mark.parametrize("fmt,prof", T.ALL_CASES, ids=CASE_IDS)
def test_samples_and_catalogue_oracle_equals_reference(fmt, prof):
    """Every sample image and the catalogue, per format and profile: the oracle's blocks equal the reference's.  Both are
    gathered from the pool results by the image's block indices (each block is encoded from its own texels alone); for
    the first five images the stored digests were recorded from whole-image runs of the reference build."""
    pl, exp = pool_for(fmt), expectation(fmt, prof)
    names = HDR_SAMPLES if fmt == "BC6H" else LDR_SAMPLES
    jobs = [(n, pl.index[n]) for n in names] + [(None, pl.catalogue_index())]
    for name, index in jobs:
        if fmt in BC45:
            key = f"bc45:{fmt}:" + (f"sample:{name}" if name else "catalogue")
        else:
            key = f"sample:{name}:{fmt}:{prof}" if name else f"catalogue:{fmt}:{prof}"
        want = reference_gathered(key, fmt, prof, index)
        assert T.same(exp[index].reshape(-1), want), key


@pytest.mark.parametrize("fmt,prof", MODE_CASES, ids=[f"{f}-{p}" for f, p in MODE_CASES])
def test_pool_reaches_every_mode(fmt, prof):
    """Mode-coverage floor: the pool's expected blocks include at least MODE_FLOOR blocks of every mode the profile emits
    (and no others), so that the mosaics below cannot quietly turn into noise."""
    m = modes(fmt, expectation(fmt, prof))
    count = {int(k): int(c) for k, c in zip(*np.unique(m, return_counts=True))}
    assert set(count) == set(EXPECTED_MODES[prof]), count
    assert min(count.values()) >= MODE_FLOOR, count


def _emu_setter(name):
    f = getattr(T.emu().lib, name)
    f.argtypes = [ctypes.c_int]
    f.restype = None
    return f


@pytest.mark.parametrize("fmt,prof", T.ALL_CASES, ids=CASE_IDS)
def test_emulation_equals_oracle_on_catalogue_and_new_samples(fmt, prof):
    """The emulated kernels on the catalogue and the images new to the suite (real alpha, a normal map, a grey ramp, a second
    HDR image); BC7 in rounds of sixteen and of eight blocks."""
    pl, exp = pool_for(fmt), expectation(fmt, prof)
    index = np.unique(np.concatenate([pl.catalogue_index()] + [pl.index[n] for n in NEW_SAMPLES if n in pl.index]))
    per_warp = _emu_setter("emu_set_bc7_per_warp")
    try:
        for pw in ((16, 8) if fmt == "BC7" else (16,)):
            per_warp(pw)
            got = encode_blocks(T.emu(), fmt, prof, pl.blocks[index])
            assert not (r := mismatch_report(got, exp[index], fmt, index, 64, pl)), f"per_warp {pw}\n{r}"
    finally:
        per_warp(16)


@pytest.mark.parametrize("fmt,prof", [("BC7", "alpha_basic"), ("BC6H", "bc6h_fast"), ("BC3", None)])
def test_emulated_mosaic_equals_gathered_expectation(fmt, prof):
    """The mosaic machinery without a GPU: a ~2 k-block mosaic through the emulated kernels equals the pool expectation
    gathered by the mosaic's permutation (layout, permutation and gathering)."""
    img, idx = mosaic(fmt, 45, 45, seed=3)
    got = T.run(T.emu(), fmt, img, prof)
    assert not (r := mismatch_report(got, expectation(fmt, prof)[idx], fmt, idx, 45, pool_for(fmt))), r


def _first_seen(pl, name, j):
    """Whether block j of source `name` is the first appearance of its pool block (so that the pool names it as its origin)."""
    k = [n for n, _, _ in pl.sources].index(name)
    p = pl.index[name][j]
    return all(p not in pl.index[n] for n, _, _ in pl.sources[:k]) and p not in pl.index[name][:j]


def test_mismatch_report_names_block_source_and_modes():
    """A result with two corrupted blocks -- one from a sample image, one from the catalogue -- is reported with each block's
    mosaic coordinate, its source and the expected and actual BC7 mode."""
    pl = pool(False)
    img_j = next(j for j in range(200, 3025) if _first_seen(pl, "monkey.png", j))
    cat_j = next(j for j in range(5, 256) if _first_seen(pl, "two-far", j))
    _, idx = mosaic("BC7", 16, 8, seed=5)
    idx = idx.copy()
    idx[16 * 3 + 5], idx[16 * 7 + 15] = pl.index["monkey.png"][img_j], pl.index["two-far"][cat_j]
    exp = expectation("BC7", "veryfast")[idx]
    got = exp.copy()
    lines = []
    for k, origin in ((16 * 3 + 5, f"monkey.png block ({img_j % 55}, {img_j // 55})"), (16 * 7 + 15, f"catalogue two-far #{cat_j}")):
        mode = bc7_mode(exp[k])
        other = 6 if mode != 6 else 1
        got[k, 0] = 1 << other                                         # the header of another mode
        lines.append(f"mosaic block ({k % 16}, {k // 16}) = pool block {idx[k]} from {origin}: mode {mode} expected, {other} got;")
    r = mismatch_report(got.reshape(-1), exp.reshape(-1), "BC7", idx, 16, pl)
    assert r.startswith("BC7: 2 of 128 blocks differ"), r
    for line in lines:
        assert line in r, (line, r)
    assert mismatch_report(exp.reshape(-1), exp.reshape(-1), "BC7", idx, 16, pl) == ""
    assert len(mismatch_report(np.zeros_like(exp), exp, "BC7", idx, 16, pl).splitlines()) == 1 + 8     # at most eight blocks


# ---------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def mosaic_shapes(fmt):
    """(width, height) in blocks, from the SM count S: BC7 one block row either side of the 8 <-> 16 round switch
    (S x 256 blocks) and a 257-wide surface of several sixteen-block rounds per CTA with ragged last round and tile; BC6H
    three rounds of 48-block tiles (both stage buffers) with a ragged tail; BC1-BC5 many CTAs with a ragged last one."""
    s = sm_count()
    if fmt == "BC7":
        return [(64, 4 * s - 1), (64, 4 * s), (257, -(-16 * s // 10))]
    if fmt == "BC6H":
        return [(257, 64)]
    return [(257, -(-16 * s // 10))]


def checked_expectation(fmt, prof):
    """The pool expectation, checked against the stored digest of the reference's pool result (the reference is not read)."""
    exp = expectation(fmt, prof)
    assert T.same(exp, T.reference(pool_key(fmt, prof), None)), "the oracle's pool result differs from the stored reference digest"
    return exp


def _seed(fmt, prof, wb, hb):
    return zlib.crc32(f"{fmt}:{prof}:{wb}x{hb}".encode())


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,prof", T.ALL_CASES, ids=CASE_IDS)
def test_gpu_sample_images_equal_reference(fmt, prof):
    """Each sample image whole through CompressBlocks* (host surfaces), against the reference's stored blocks."""
    lib = T.product()
    for name in (HDR_SAMPLES if fmt == "BC6H" else LDR_SAMPLES):
        img = sample(name)
        key = f"bc45:{fmt}:sample:{name}" if fmt in BC45 else f"sample:{name}:{fmt}:{prof}"
        got = lib.encode(fmt, img, lib.profile(prof) if prof else None)
        assert T.same(got, T.reference(key, None)), key


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,prof", T.ALL_CASES, ids=CASE_IDS)
def test_gpu_mosaics_every_entry_point(fmt, prof):
    """Mosaics through: device source and destination (one launch of the TMA / vector-load kernels); a device source offset
    off 16-byte alignment (+4 bytes RGBA8, +8 RGBA16F: the plain-load kernels); host pageable memory (the banded pipeline for
    BC7 / BC6H)."""
    import torch
    lib = T.product()
    exp = checked_expectation(fmt, prof)
    settings = lib.profile(prof) if prof else None
    _, bpb, texel, _ = T.binding.FORMATS[fmt]
    pl = pool_for(fmt)
    for wb, hb in mosaic_shapes(fmt):
        img, idx = mosaic(fmt, wb, hb, _seed(fmt, prof, wb, hb))
        want = exp[idx]
        w, h = 4 * wb, 4 * hb
        raw = img.view(np.uint8).reshape(-1)
        for shift in (0, texel):
            d_in = torch.zeros(raw.size + 16, dtype=torch.uint8, device="cuda")
            d_in[shift:shift + raw.size] = torch.from_numpy(raw).cuda()
            d_out = torch.zeros(wb * hb * bpb, dtype=torch.uint8, device="cuda")
            lib.encode_raw(fmt, d_in.data_ptr() + shift, w, h, w * texel, d_out.data_ptr(), settings)
            torch.cuda.synchronize()
            r = mismatch_report(d_out.cpu().numpy(), want, fmt, idx, wb, pl)
            assert not r, f"{wb}x{hb} blocks, device source +{shift} bytes\n{r}"
        r = mismatch_report(lib.encode(fmt, img, settings), want, fmt, idx, wb, pl)
        assert not r, f"{wb}x{hb} blocks, host pageable\n{r}"


STREAM_CASES = [("BC1", None), ("BC3", None), ("BC4", None), ("BC5", None), ("BC7", "alpha_slow"), ("BC6H", "bc6h_veryslow")]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,prof", STREAM_CASES, ids=[f"{f}-{p}" for f, p in STREAM_CASES])
def test_gpu_mosaic_on_caller_stream(fmt, prof):
    """itw_encode_device on a non-default stream, the largest mosaic of the format."""
    import torch
    lib = T.product()
    exp = checked_expectation(fmt, prof)
    _, bpb, texel, _ = T.binding.FORMATS[fmt]
    wb, hb = mosaic_shapes(fmt)[-1]
    img, idx = mosaic(fmt, wb, hb, _seed(fmt, prof, wb, hb) + 1)
    d_in = torch.from_numpy(img.view(np.uint8).reshape(-1)).cuda()
    d_out = torch.zeros(wb * hb * bpb, dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        lib.encode_device(fmt, d_in.data_ptr(), 4 * wb, 4 * hb, 4 * wb * texel, d_out.data_ptr(),
                          lib.profile(prof) if prof else None, s.cuda_stream)
    s.synchronize()
    assert not (r := mismatch_report(d_out.cpu().numpy(), exp[idx], fmt, idx, wb, pool_for(fmt))), r


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,prof", [("BC1", None), ("BC7", "basic"), ("BC6H", "bc6h_basic")])
def test_gpu_mosaic_fanned_out_over_devices(fmt, prof):
    """Host calls fanned out over every visible GPU (itw_set_devices), the largest mosaic of the format."""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"fan-out needs two or more visible GPUs; {n} visible")
    lib = T.product()
    exp = checked_expectation(fmt, prof)
    wb, hb = mosaic_shapes(fmt)[-1]
    img, idx = mosaic(fmt, wb, hb, _seed(fmt, prof, wb, hb) + 2)
    lib.set_devices(list(range(n)))
    try:
        got = lib.encode(fmt, img, lib.profile(prof) if prof else None)
    finally:
        lib.set_devices([])
    assert not (r := mismatch_report(got, exp[idx], fmt, idx, wb, pool_for(fmt))), r
