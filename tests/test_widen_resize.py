"""vips_resize with VIPS_KERNEL_NEAREST when the shrink is large enough for resize.c:167-205 to subsample first
(vips_subsample: the integer part of the shrink over gap), then reduce the residual.

Found by a random oracle-vs-reference campaign over sizes / scales / kernels / formats (the only disagreement in 15 000
cases): the oracle used to reduce by the whole factor in one go, which picks other pixels and sometimes another size.
CPU: the oracle, now with the subsample step, against the reference's own resize.c + subsample.c + reducev / reduceh under
oracle/_ref.  GPU: the device path has no subsample step and must decline these calls (the host keeps its C path) instead of
computing something else."""
import numpy as np
import pytest

from oracle import pyoracle as orc
from oracle import pyref
from refgold import ref  # noqa: F401

CASES = [(186, 101, 0.125, 0.125), (72, 169, 0.08, 0.295), (165, 147, 1 / 6, 0.3777), (104, 178, 0.0832, 0.0832),
         (198, 178, 0.125, 0.125), (28, 50, 1 / 7, 1 / 7), (300, 200, 0.05, 0.9), (64, 64, 0.25, 0.25), (65, 63, 0.26, 0.24)]


def test_oracle_nearest_resize_subsamples_like_the_reference(ref):
    rng = np.random.default_rng(5)
    for (w, h, sc, vs) in CASES:
        for dt in (np.uint8, np.int16, np.float32):
            a = (rng.random((h, w, 3)) * 200).astype(dt)
            got = orc.resize(a, sc, vs, "nearest")
            ref.check(got, lambda: pyref.RefImage.from_array(a).resize(sc, vs, "nearest").numpy(), (w, h, sc, vs, dt))
    # gap < 1: the integer part of 1 / scale, not of size / target / gap (resize.c:173-176)
    a = rng.integers(0, 256, (90, 120, 1), dtype=np.uint8)
    for gap in (0.0, 0.5, 1.0, 3.0):
        ref.check(orc.resize(a, 0.2, 0.3, "nearest", gap), lambda: pyref.RefImage.from_array(a).resize(0.2, 0.3, "nearest", gap).numpy(), gap)

    # subsample.c itself: out(x, y) = in(x * xfac, y * yfac), size rounded down
    def subsample():
        L = pyref.lib()
        L.ref_subsample.restype = __import__("ctypes").c_void_p
        L.ref_subsample.argtypes = [__import__("ctypes").c_void_p, __import__("ctypes").c_int, __import__("ctypes").c_int]
        im = pyref.RefImage.from_array(a)
        return pyref.RefImage(L.ref_subsample(im.h, 7, 4), (im,)).numpy()
    ref.check(a[:88:4, :119:7][:90 // 4, :120 // 7], subsample)


@pytest.mark.gpu
def test_gpu_nearest_resize_declines_the_subsample_cases(vb):
    rng = np.random.default_rng(6)
    a = rng.integers(0, 256, (101, 186, 3), dtype=np.uint8)
    with pytest.raises(vb.Error, match="subsample step"):
        vb.Image(a).resize(0.125, kernel="nearest")
    with pytest.raises(vb.Error, match="subsample step"):
        vb.Image(a).resize(0.9, 0.05, kernel="nearest")
