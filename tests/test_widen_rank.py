"""vips_rank / vips_median (SURVEY 8f rank 4).  CPU: the oracle against the reference's own morphology/rank.c under
oracle/_ref (histogram, select, max and min paths, tiled and untiled), the kernel's staging + radix-select code
compiled for the host (vb200_debug_rank_host) against the oracle, and the reference test-suite's known answer.
GPU: rank_kernel against the oracle, bit for bit."""
import numpy as np
import pytest

from oracle import pyconv, pyref
from refgold import ref  # noqa: F401

DTYPES = (np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32)
# (width, height, index): median 3x3 / 5x5, min, max, the uchar histogram path (n > 90 and n > 10 mid-index), odd shapes
WINDOWS = [(3, 3, 4), (3, 3, 0), (3, 3, 8), (5, 5, 12), (5, 3, 7), (1, 1, 0), (11, 11, 50), (4, 4, 3), (10, 10, 99), (2, 7, 5),
           (1, 6, 2), (9, 1, 8)]


def image(rng, dt, shape):
    if np.dtype(dt).kind == "f":
        return ((rng.random(shape) - 0.5) * 1000).astype(dt)
    info = np.iinfo(dt)
    lo, hi = max(info.min, -2 ** 31), min(info.max, 2 ** 32 - 1)
    a = rng.integers(lo, hi + 1, shape, dtype=np.int64).astype(dt)
    a[rng.random(shape) < 0.3] = a.flat[0]  # ties
    return a


def test_oracle_rank_matches_reference(ref):
    rng = np.random.default_rng(11)
    for dt in DTYPES:
        a = image(rng, dt, (37, 45, 3))
        for (rw, rh, idx) in WINDOWS:
            got = pyconv.rank(a, rw, rh, idx)
            ref.check(got, lambda: pyconv.ref_rank(a, rw, rh, idx), (dt, rw, rh, idx))
            ref.check(got, lambda: pyconv.ref_rank(a, rw, rh, idx, tile=(16, 16)), (dt, rw, rh, idx))


def test_host_twin_matches_oracle():
    import libvips_b200 as vb
    rng = np.random.default_rng(12)
    for dt in DTYPES:
        for shape in ((37, 45, 3), (9, 70, 1), (41, 33, 4), (12, 12, 5)):
            a = image(rng, dt, shape)
            for (rw, rh, idx) in WINDOWS:
                if rw > shape[1] or rh > shape[0]:
                    continue
                assert np.array_equal(vb.rank_host_twin(a, rw, rh, idx), pyconv.rank(a, rw, rh, idx)), (dt, shape, rw, rh, idx)
    # special floats: infinities and signed zeros order as numbers (-0 < +0 by bit pattern)
    f = np.array([[np.inf, -np.inf, 0.0], [-0.0, 1e-45, -1e-45], [3.0, -3.0, 1e38]], np.float32)[:, :, None]
    for idx in range(9):
        got = vb.rank_host_twin(f, 3, 3, idx)[1, 1, 0]
        want = np.sort(f.ravel())[idx]
        assert got == want, (idx, got, want)
    # a window that does not fit the default 32 x 8 tile in shared memory: the plan shrinks the tile
    a = image(rng, np.uint32, (70, 300, 4))
    assert np.array_equal(vb.rank_host_twin(a, 61, 61, 1000), pyconv.rank(a, 61, 61, 1000))
    with pytest.raises(vb.Error, match="window too large"):
        vb.rank_host_twin(np.zeros((4, 4, 1), np.uint8), 5, 3, 0)
    with pytest.raises(vb.Error, match="index out of range"):
        vb.rank_host_twin(np.zeros((4, 4, 1), np.uint8), 3, 3, 9)


def test_known_answers():
    """test/test-suite/test_morphology.py:44-51 (test_rank): a filled white circle of radius 25 on black under rank(3, 3, 8)
    -- the window's maximum -- keeps its geometry and gets brighter on average; plus what follows from the definition: a
    10 x 10 square grows by one pixel on every side, the median of a constant image is the constant"""
    yy, xx = np.mgrid[0:100, 0:100]
    im = (((xx - 50) ** 2 + (yy - 50) ** 2 <= 25 * 25) * 255).astype(np.uint8)[:, :, None]
    im2 = pyconv.rank(im, 3, 3, 8)
    assert im2.shape == im.shape and im2.mean() > im.mean()
    sq = np.zeros((100, 100, 1), np.uint8)
    sq[45:55, 45:55] = 255
    sq2 = pyconv.rank(sq, 3, 3, 8)
    assert sq2[44:56, 44:56].min() == 255 and sq2.sum() == 144 * 255
    assert np.array_equal(pyconv.median(np.full((20, 20, 3), 7, np.uint8), 5), np.full((20, 20, 3), 7, np.uint8))
    with pytest.raises(ValueError):
        pyconv.rank(sq, 3, 3, 9)


@pytest.mark.gpu
def test_gpu_rank(vb):
    rng = np.random.default_rng(13)
    for dt in DTYPES:
        for shape in ((37, 45, 3), (130, 261, 4), (64, 64, 1)):
            a = image(rng, dt, shape)
            for (rw, rh, idx) in WINDOWS:
                got = vb.Image(a).rank(rw, rh, idx).numpy()
                assert np.array_equal(got, pyconv.rank(a, rw, rh, idx)), (dt, shape, rw, rh, idx)
    a = image(rng, np.uint8, (300, 517, 3))
    assert np.array_equal(vb.Image(a).median(3).numpy(), pyconv.median(a, 3))
    # large window (tile shrinks, opt-in shared memory)
    a = image(rng, np.uint32, (70, 300, 4))
    assert np.array_equal(vb.Image(a).rank(61, 61, 1000).numpy(), pyconv.rank(a, 61, 61, 1000))
    with pytest.raises(vb.Error, match="index out of range"):
        vb.Image(np.zeros((8, 8, 1), np.uint8)).rank(3, 3, 9)
    # in a chain: median then dilate
    m = np.full((3, 3), 255.0)
    b = (rng.random((90, 120, 1)) > 0.4).astype(np.uint8) * 255
    got = vb.Chain().rank(3, 3, 4).morph(m, "dilate").run([b])[0].numpy()
    assert np.array_equal(got, pyconv.morph(pyconv.median(b, 3), m, "dilate"))
