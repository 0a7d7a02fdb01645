"""Writes tests/golden/refgpu_digests.json: sha256 digests (refgpu.digest) of the CPU oracle's
outputs for every input tests/test_gpu_reference.py and
tests/test_gpu_factored.py::test_default_u8_against_the_compiled_reference compare against.
They stand in for the reference kernels' outputs, so those comparisons run on any machine,
whether or not the reference is built into oracle/_ref.

The reference's outputs at these sizes do not fit in the repository and its sources do not
ship with it, so the digests are the ORACLE's.  Before writing, this script checks the oracle
bit for bit against the reference outputs committed as tests/golden/refgpu_*.npz (up to
128x128) and against SURVEY.md Appendix B's known answers (sums and counts at 256^2, 1024^2 and
8192^2).  The full-size digests themselves are compared with the reference only where
oracle/_ref is built: the tests then check every digest they use against the live reference.

    python tests/golden/make_ref_digests.py
"""
import glob
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import inputs  # noqa: E402
import refgpu  # noqa: E402
from oracle import oracle as o  # noqa: E402

THREADS = max(1, min(8, os.cpu_count() or 1))
APPENDIX_B = {256: (-306, 114414, 46317, 8329775), 1024: (-2562, 1831230, 741557, 133161285),
              8192: (-268447, 117045095, 47462419, 8524699637)}


def check_oracle_is_the_reference():
    files = sorted(glob.glob(os.path.join(HERE, "refgpu_*.npz")))
    assert files, "no reference fixtures"
    for f in files:
        g = np.load(f)
        coef, shifted = o.dct(g["img"].astype(np.float32), want_shifted=True)
        assert np.array_equal(coef.view(np.uint32), g["coef"].view(np.uint32)), f
        assert np.array_equal(shifted, g["shifted"]), f
        assert np.array_equal(o.idct(coef).view(np.uint32), g["rec"].view(np.uint32)), f


def transform(img, Q=None):
    coef, shifted = o.dct(img, Q=Q, want_shifted=True, threads=THREADS)
    return coef, shifted, o.idct(coef, Q=Q, threads=THREADS)


def main():
    o.build()
    check_oracle_is_the_reference()
    cases = {}
    # the reference benchmark's input (srand(42); rand()%256), Haweel T, JPEG Q
    for N in (256, 512, 1024, 2048, 8192):
        img = o.rand_image(N, N, 42)
        coef, shifted, rec = transform(img)
        u8 = o.to_u8(rec)
        if N in APPENDIX_B:
            got = (int(coef.sum(dtype=np.float64)), int(np.abs(coef).sum(dtype=np.float64)),
                   int(np.count_nonzero(coef)), int(u8.sum(dtype=np.int64)))
            assert got == APPENDIX_B[N], (N, got)
        mse, peen = o.metrics(img.astype(np.uint8), u8)
        cases[f"rand{N}"] = {"coef": refgpu.digest(coef), "shifted": refgpu.digest(shifted),
                             "rec": refgpu.digest(rec), "mse": mse, "peen": peen}
    for name, img in (("adversarial32", inputs.adversarial(32)), ("floatnoise64x256", inputs.float_noise(64, 256)),
                      ("rand48x640_seed7", o.rand_image(48, 640, 7))):
        coef, shifted, rec = transform(img)
        cases[name] = {"coef": refgpu.digest(coef), "shifted": refgpu.digest(shifted), "rec": refgpu.digest(rec)}
    coef, shifted, rec = transform(o.rand_image(256, 256, 5), Q=o.jpeg_Q() * 0.5)
    cases["rand256_seed5_halfq"] = {"coef": refgpu.digest(coef), "shifted": refgpu.digest(shifted), "rec": refgpu.digest(rec)}
    # the reference's own u8 flow: u8 image -> float -> DCT -> IDCT -> clamp and truncate to u8
    for N in (2048, 8192):
        img8 = o.rand_image_u8(N, N, 42)
        coef, _, rec = transform(img8.astype(np.float32))
        u8 = o.to_u8(rec)
        mse, peen = o.metrics(img8, u8)
        cases[f"u8flow{N}"] = {"coef_i16": refgpu.digest(coef.astype(np.int16)), "u8": refgpu.digest(u8),
                               "mse": mse, "peen": peen}
    doc = {"what": "sha256 digests (tests/refgpu.py digest()) of the CPU oracle's outputs, which equal the reference "
                   "kernels' on tests/golden/refgpu_*.npz and SURVEY.md Appendix B; written by "
                   "tests/golden/make_ref_digests.py", "cases": cases}
    with open(refgpu.DIGESTS, "w") as f:
        json.dump(doc, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", refgpu.DIGESTS, len(cases), "cases")


if __name__ == "__main__":
    main()
