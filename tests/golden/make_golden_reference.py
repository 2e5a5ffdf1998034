#!/usr/bin/env python3
"""Generate tests/golden/reference_digests.json: the digest (tests/itw_testlib.py digest()) of every result the tests
take from the reference's own code -- the reference-source builds under oracle/_ref and the tables of the reference
checkout -- so that the same comparisons run where neither is available.

Run after build(), with the path of a reference checkout:   python tests/golden/make_golden_reference.py <reference checkout>

The CPU tests that compare with the reference run once with recording on (tests/itw_testlib.py reference()); the
reference results that only GPU tests compare against are computed here directly."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
OUT = os.path.join(HERE, "reference_digests.json")
CPU_TESTS = ["test_abi.py", "test_bc45_vs_directxtex.py", "test_dds.py", "test_decode.py", "test_decode_vs_directxtex.py",
             "test_frontend.py", "test_kat.py", "test_mips.py", "test_mips_f16.py", "test_oracle_vs_ref.py", "test_random_settings.py",
             "test_real_content.py", "test_tables.py", "test_gpu_content.py", "test_gpu_prepass.py"]


def record_gpu_only():
    sys.path.insert(0, TESTS)
    import itw_testlib as T
    import test_decode_vs_directxtex as DV
    import test_full_configs as F
    from test_decode import random_blocks
    assert T.ref() is not None, "needs oracle/_ref (build() with the reference checkout present)"
    for name, fmt, prof, surfaces in F.G.configs():
        img = T.synth.mixed_rgba8(8192, 8192) if name == "C4" else surfaces[0]     # C4 checks level 0 of the GPU-made chain
        F.reference_rows(name, fmt, prof, img, F.LIVE_STEP[name])
    for fid, base in ((98, "BC7"), (95, "BC6H"), (96, "BC6H")):
        DV.dx_decode(DV.dx(), fid, random_blocks(base, 256 * 256, seed=77), "random-bits-large")


def main(reference_root):
    env = dict(os.environ, ITW_RECORD_REFERENCE=OUT, ITW_REFERENCE_ROOT=os.path.abspath(reference_root))
    if os.path.exists(OUT):
        os.remove(OUT)
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", "-m", "not gpu"]
                          + [os.path.join(TESTS, t) for t in CPU_TESTS], cwd=os.path.dirname(TESTS), env=env)
    subprocess.check_call([sys.executable, os.path.abspath(__file__), "--gpu-only"], env=env)


if __name__ == "__main__":
    if sys.argv[1] == "--gpu-only":
        record_gpu_only()
    else:
        main(sys.argv[1])
