"""Real-content check (SURVEY.md 8d): the reference's own sample images through the reference-source build, the oracle and
the emulated kernels.  The crops the test encodes are stored as tests/golden/sample_images.npz (made by
tests/golden/make_golden_samples.py from the reference's "Sample Images"); the reference build's blocks come from
oracle/_ref where it is built and from their stored digests elsewhere."""
import os

import numpy as np
import pytest

import itw_testlib as T

SAMPLES = os.path.join(os.path.dirname(__file__), "golden", "sample_images.npz")


def load(name):
    with np.load(SAMPLES) as z:
        return np.ascontiguousarray(z[name])


LDR = [("baboon.png", (64, 64, 128, 128)), ("gradients.png", None), ("colors-260K.png", (128, 128, 128, 128)), ("colors-16M.png", (1024, 2048, 64, 128)),
       ("juggling-balls.jpg", (200, 300, 128, 128))]


@pytest.mark.parametrize("name,crop", LDR)
def test_ldr_samples_reference_build_oracle_and_emulated_kernels_agree(name, crop):
    ref, o, e = T.ref(), T.oracle(), T.emu()
    img = load(name)
    if crop:
        assert img.shape[:2] == crop[2:], name
    for fmt, prof in (("BC1", None), ("BC3", None), ("BC7", "slow"), ("BC7", "alpha_basic"), ("BC7", "veryfast")):
        want = T.reference(f"sample:{name}:{fmt}:{prof}", ref and (lambda: T.run(ref, fmt, img, prof)))
        assert T.same(T.run(o, fmt, img, prof), want), (name, fmt, prof, "oracle")
        assert T.same(T.run(e, fmt, img, prof), want), (name, fmt, prof, "emulated kernel")
    for fmt in ("BC4", "BC5"):
        assert np.array_equal(T.run(e, fmt, img, None), T.run(o, fmt, img, None)), (name, fmt)


def test_hdr_sample_reference_build_oracle_and_emulated_kernel_agree():
    ref, o, e = T.ref(), T.oracle(), T.emu()
    img = load("HDR.hdr")                                                # rows and columns 64..191 of HDR.hdr
    assert img.shape == (128, 128, 4)
    assert len(np.unique(img[..., :3])) > 300                            # a real HDR crop, not a flat region
    for prof in ("bc6h_slow", "bc6h_basic", "bc6h_veryfast"):
        want = T.reference(f"sample:HDR.hdr:BC6H:{prof}", ref and (lambda: T.run(ref, "BC6H", img, prof)))
        assert T.same(T.run(o, "BC6H", img, prof), want), prof
        assert T.same(T.run(e, "BC6H", img, prof), want), prof
