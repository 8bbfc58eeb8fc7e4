"""vips_morph (SURVEY 8f rank 4).  CPU: the oracle against the reference's own morphology/morph.c under oracle/_ref and
the reference test-suite's known answers (test_morphology.py: erode / dilate of a dot with a cross).  GPU: the CUDA
kernel against the oracle, bit for bit."""
import numpy as np
import pytest

from oracle import pyconv, pyref
from refgold import ref  # noqa: F401

MASKS = [np.array([[128, 255, 128], [255, 255, 255], [128, 255, 128]], np.float64),
         np.array([[255, 255, 255], [255, 255, 255], [255, 255, 255]], np.float64),
         np.array([[0, 255, 128, 255, 0]], np.float64),
         np.array([[255], [128], [0], [255]], np.float64),
         np.full((7, 5), 255.0)]


def images(rng):
    binary = (rng.random((61, 83, 1)) > 0.6).astype(np.uint8) * 255
    grey = rng.integers(0, 256, (40, 57, 3), dtype=np.uint8)  # the ops are bitwise: any byte values
    return [binary, grey, rng.integers(0, 256, (5, 3, 4), dtype=np.uint8)]


def test_oracle_morph_matches_reference(ref):
    rng = np.random.default_rng(3)
    for a in images(rng):
        for m in MASKS:
            for op in ("erode", "dilate"):
                got = pyconv.morph(a, m, op)
                ref.check(got, lambda: pyconv.ref_morph(a, m, op), (a.shape, m.shape, op))
                ref.check(got, lambda: pyconv.ref_morph(a, m, op, tile=(16, 16)), (a.shape, m.shape, op))


def test_known_answers():
    """test/test-suite/test_morphology.py: a white dot eroded by a cross vanishes, dilated becomes the cross"""
    im = np.zeros((100, 100, 1), np.uint8)
    im[45:55, 45:55] = 255
    cross = MASKS[0]
    e = pyconv.morph(im, cross, "erode")
    d = pyconv.morph(im, cross, "dilate")
    assert e.sum() < im.sum() < d.sum()
    assert e[50, 50, 0] == 255 and e[45, 45, 0] == 0 and d[44, 50, 0] == 255 and d[44, 44, 0] == 0
    with pytest.raises(ValueError):
        pyconv.morph(im, np.array([[1.0, 255.0]]), "erode")


@pytest.mark.gpu
def test_gpu_morph(vb):
    rng = np.random.default_rng(4)
    for a in images(rng) + [rng.integers(0, 256, (300, 517, 3), dtype=np.uint8)]:
        for m in MASKS:
            for op in ("erode", "dilate"):
                got = vb.Image(a).morph(m, op).numpy()
                assert np.array_equal(got, pyconv.morph(a, m, op)), (a.shape, m.shape, op)
    with pytest.raises(vb.Error, match="should be 0, 128 or 255"):
        vb.Image(np.zeros((8, 8, 1), np.uint8)).morph(np.array([[7.0]]), "erode")
    # in a chain: open = erode then dilate
    a = (rng.random((90, 120, 1)) > 0.4).astype(np.uint8) * 255
    got = vb.Chain().morph(MASKS[1], "erode").morph(MASKS[1], "dilate").run([a])[0].numpy()
    assert np.array_equal(got, pyconv.morph(pyconv.morph(a, MASKS[1], "erode"), MASKS[1], "dilate"))
