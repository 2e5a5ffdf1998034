"""Partition ("shape") tables: the device header, the oracle's compact arrays, kernel.ispc's packed tables and
DirectXTex's canonical g_aPartitionTable / g_aFixUp must all describe the same 128 shapes.  The reference's tables are
read from its checkout where one is present, and compared through their stored digests elsewhere."""
import hashlib
import os
import re

import numpy as np

import itw_testlib as T

CSRC = os.path.join(T.ROOT, "intel-texture-works-plugin_b200", "csrc")
REF = os.environ.get("ITW_REFERENCE_ROOT", "/root/reference")
TABLE_DIGEST = "6c4572d3d53dd54f"      # first 16 hex of sha256 over (pattern, anchors) -- see test below


def device_tables():
    src = open(os.path.join(CSRC, "itw_tables.cuh")).read()

    def grab(name):
        m = re.search(r"#define ITW_TABLE_INIT_" + name + r" \\\n(.*?)\n\n", src, re.S)
        return [int(x.rstrip("u"), 0) for x in re.findall(r"0x[0-9A-Fa-f]+u?|\b\d+\b", m.group(1))]
    return grab("shape_pattern"), grab("shape_mask01"), grab("shape_anchor1"), grab("shape_anchor2")


def oracle_tables():
    src = open(os.path.join(T.ROOT, "oracle", "itw_oracle.cpp")).read()

    def arr(name):
        m = re.search(name + r"\[64\]\s*=\s*\{(.*?)\};", src, re.S)
        return [int(x, 0) for x in re.findall(r"0x[0-9A-Fa-f]+|\b\d+\b", m.group(1))]
    pat = []
    for m in arr("kShape2"):
        pat.append(sum(((m >> k) & 1) << (2 * k) for k in range(16)))
    pat += arr("kShape3")
    return pat, arr("kAnchor2") + arr("kAnchor3a"), [0] * 64 + arr("kAnchor3b")


def test_device_tables_self_consistent_and_equal_to_oracle():
    pat, mask, a1, a2 = device_tables()
    assert [len(x) for x in (pat, mask, a1, a2)] == [128] * 4
    for i in range(128):
        subsets = [(pat[i] >> (2 * k)) & 3 for k in range(16)]
        assert max(subsets) == (1 if i < 64 else 2)
        assert subsets[0] == 0                                   # texel 0 always anchors subset 0
        m0 = sum(1 << k for k in range(16) if subsets[k] == 0)
        m1 = sum(1 << k for k in range(16) if subsets[k] == 1)
        assert mask[i] == (m0 | (m1 << 16))
        assert subsets[a1[i]] == 1                               # anchors lie in their own subset ...
        if i >= 64:
            assert subsets[a2[i]] == 2
    opat, oa1, oa2 = oracle_tables()
    assert opat == pat and oa1 == a1 and oa2 == a2
    blob = ",".join(map(str, pat + a1 + a2)).encode()
    assert hashlib.sha256(blob).hexdigest()[:16] == TABLE_DIGEST    # pinned when checked against the reference


def test_anchor_is_first_texel_of_subset_in_the_spec_sense():
    """BC7 anchors are the FIRST texel of each subset in raster order for most shapes, but not all
    (the spec lists them explicitly); check the defining property that does hold for every shape:
    the anchor belongs to its subset, and subset 0's anchor is texel 0."""
    pat, _, a1, a2 = device_tables()
    for i in range(128):
        assert (pat[i] >> (2 * a1[i])) & 3 == 1
        if i >= 64:
            assert (pat[i] >> (2 * a2[i])) & 3 == 2


def _read_reference(*parts):
    """A file of the reference checkout, or None where it is not present (the stored digests stand in)."""
    path = os.path.join(REF, *parts)
    return open(path, encoding="utf-8", errors="replace").read() if os.path.exists(path) else None


def test_tables_equal_reference_kernel_and_directxtex():
    pat, mask, a1, a2 = device_tables()
    k = _read_reference("IntelCompressionPlugin", "kernel.ispc")

    def ktab(name):
        m = re.search(name + r"\[\]\s*=\s*\{(.*?)\};", k, re.S)
        return np.array([int(x.rstrip("u"), 16) for x in re.findall(r"0x[0-9a-fA-F]+u?", m.group(1))], np.int64)

    def ref(key, compute):
        return T.reference(f"tables:{key}", k and d and compute)
    d = _read_reference("3rdParty", "DirectXTex", "DirectXTex", "BC6HBC7.cpp")
    assert T.same(np.array(pat, np.int64), ref("kernel.ispc:pattern_table", lambda: ktab("pattern_table")))              # kernel.ispc:690-707
    assert T.same(np.array(mask, np.int64), ref("kernel.ispc:pattern_mask_table", lambda: ktab("pattern_mask_table")))   # kernel.ispc:714-731
    # kernel.ispc:743-752: anchor 1 in the high nibble of skip_table, anchor 2 (three-subset shapes) in the low one
    assert T.same(np.array(a1, np.int64), ref("kernel.ispc:skip_table>>4", lambda: ktab("skip_table") >> 4))
    assert T.same(np.array(a2[64:], np.int64), ref("kernel.ispc:skip_table[64:]&15", lambda: ktab("skip_table")[64:] & 15))

    def partitions():
        body = d[d.index("g_aPartitionTable[3][64][16]"):d.index("g_aFixUp[3][64][3]")]
        rows = re.findall(r"\{((?:\s*\d\s*,){15}\s*\d\s*)\}", body)
        assert len(rows) == 192
        return np.array([[int(x) for x in r.split(",")] for r in rows[64:]], np.int64)     # DirectXTexBC6HBC7.cpp:40 (2- and 3-subset tables)
    want = np.array([[(p >> (2 * i)) & 3 for i in range(16)] for p in pat], np.int64)
    assert T.same(want, ref("BC6HBC7.cpp:g_aPartitionTable[1:]", partitions))

    def fixups():
        fix = d[d.index("g_aFixUp[3][64][3]"):]
        trip = re.findall(r"\{\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*\}", fix[:fix.index("};")])
        assert len(trip) == 192
        return np.array([int(t[1]) for t in trip[64:]] + [int(t[2]) for t in trip[128:]], np.int64)   # DirectXTex BC6HBC7.cpp:247
    assert T.same(np.array(a1 + a2[64:], np.int64), ref("BC6HBC7.cpp:g_aFixUp[1:]", fixups))


def test_weight_formula_equals_the_spec_tables():
    """csrc/itw_device.cuh computes BC7 weights arithmetically; it must reproduce kernel.ispc:679-681."""
    tables = {2: [0, 21, 43, 64], 3: [0, 9, 18, 27, 37, 46, 55, 64], 4: [0, 4, 9, 13, 17, 21, 26, 30, 34, 38, 43, 47, 51, 55, 60, 64]}
    mult = {2: 5462, 3: 2341, 4: 1093}
    src = open(os.path.join(CSRC, "itw_device.cuh")).read()
    assert "5462" in src and "2341" in src and "1093" in src
    for bits, tab in tables.items():
        n = (1 << bits) - 1
        assert [((64 * q + (n >> 1)) * mult[bits]) >> 14 for q in range(n + 1)] == tab
