#!/usr/bin/env python3
"""Generate tests/golden/sample_images.npz: the crops of the reference's own sample images that tests/test_real_content.py and
tests/test_gpu_content.py encode, decoded to the surfaces the encoders take (RGBA8, and RGBA16F half bits for the Radiance
HDR files).  monkey.png brings a real 0..255 alpha channel, normals.png a normal map (BC5's input), radial-grayscale.png a
smooth single channel (BC4's input).  New images are only ever appended: the stored reference digests cover the old ones.

Run with the path of a reference checkout:   python tests/golden/make_golden_samples.py <reference checkout>
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "sample_images.npz")

# (file, crop (y, x, h, w) or None for the whole image)
LDR = [("baboon.png", (64, 64, 128, 128)), ("gradients.png", None), ("colors-260K.png", (128, 128, 128, 128)), ("colors-16M.png", (1024, 2048, 64, 128)),
       ("juggling-balls.jpg", (200, 300, 128, 128)), ("monkey.png", None), ("normals.png", None), ("radial-grayscale.png", None)]
HDR = [("HDR.hdr", (64, 64, 128, 128)), ("monkey-32bit.hdr", None)]


def load_rgba8(samples, name, crop=None):
    from PIL import Image
    img = np.array(Image.open(os.path.join(samples, name)).convert("RGBA"))
    if crop:
        y, x, h, w = crop
        img = img[y:y + h, x:x + w]
    h, w = (img.shape[0] // 4) * 4, (img.shape[1] // 4) * 4
    return np.ascontiguousarray(img[:h, :w])


def load_radiance_hdr(samples, name, crop=None):
    """Minimal Radiance RGBE reader (new-style RLE scanlines) -> RGBA16F half bits; crop (y, x, h, w) or None for all of it."""
    data = open(os.path.join(samples, name), "rb").read()
    pos = data.index(b"\n\n") + 2
    end = data.index(b"\n", pos)
    tokens = data[pos:end].split()
    assert tokens[0] == b"-Y" and tokens[2] == b"+X", tokens
    h, w = int(tokens[1]), int(tokens[3])
    pos = end + 1
    rows = []
    y0, x0, ch, cw = crop or (0, 0, h, w)
    for y in range(min(h, y0 + ch)):
        assert data[pos] == 2 and data[pos + 1] == 2 and ((data[pos + 2] << 8) | data[pos + 3]) == w
        pos += 4
        line = np.zeros((4, w), np.uint8)
        for c in range(4):
            x = 0
            while x < w:
                n = data[pos]
                pos += 1
                if n > 128:
                    line[c, x:x + n - 128] = data[pos]
                    pos += 1
                    x += n - 128
                else:
                    line[c, x:x + n] = np.frombuffer(data[pos:pos + n], np.uint8)
                    pos += n
                    x += n
        if y >= y0:
            rows.append(line[:, x0:x0 + cw].copy())
    rgbe = np.stack(rows).transpose(0, 2, 1).astype(np.float32)              # H x W x 4
    scale = np.where(rgbe[..., 3] > 0, np.exp2(rgbe[..., 3] - 136.0), 0.0).astype(np.float32)
    rgb = rgbe[..., :3] * scale[..., None]
    out = np.zeros(rgb.shape[:2] + (4,), np.float16)
    out[..., :3] = np.clip(rgb, 0, 65504).astype(np.float16)
    out[..., 3] = 1.0
    out = out[:(out.shape[0] // 4) * 4, :(out.shape[1] // 4) * 4]
    return np.ascontiguousarray(out.view(np.uint16))


def main(reference_root):
    samples = os.path.join(reference_root, "Sample Images")
    arrays = {name: load_rgba8(samples, name, crop) for name, crop in LDR}
    for name, crop in HDR:
        arrays[name] = load_radiance_hdr(samples, name, crop)
    np.savez_compressed(OUT, **arrays)
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
