"""OpenCV's edge-aware demosaic (`cv2.cvtColor(uint16 mosaic, cv2.COLOR_BayerBG2RGB_EA)`, the routine behind the reference's
demosaic_CV2) on seeded mosaics: full 14-bit range, tiny ranges (gradient ties everywhere), a constant image, the smallest legal
size.  The seed and the sizes are stored with the CRC-32 of each RGB output; the test regenerates the mosaics from them.

    python tests/golden/make_golden_demosaic.py        # needs opencv-python
"""
import os
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SEED = 5
CASES = [(4, 4, 16384), (6, 10, 16384), (64, 96, 16384), (66, 130, 8), (32, 34, 2), (30, 62, 3), (128, 258, 16384)]
FLAT = (8, 12, 16383)  # constant mosaic at the 14-bit white level


def mosaics():
    """The seeded mosaics, then the constant one."""
    rng = np.random.default_rng(SEED)
    out = [rng.integers(0, hi, size=(h, w), dtype=np.uint16) for (h, w, hi) in CASES]
    return out + [np.full(FLAT[:2], FLAT[2], np.uint16)]


def crc(a):
    return np.uint32(zlib.crc32(np.ascontiguousarray(a).tobytes()))


def main():
    import cv2
    crcs = np.array([crc(cv2.cvtColor(b, cv2.COLOR_BayerBG2RGB_EA)) for b in mosaics()], np.uint32)
    np.savez_compressed(os.path.join(HERE, "demosaic_cv2.npz"), cv2_version=cv2.__version__, seed=SEED, cases=np.array(CASES),
                        flat=np.array(FLAT), crc=crcs)
    print(cv2.__version__, crcs.tolist())


if __name__ == "__main__":
    main()
