"""Convolution path.  CPU: the oracle against the reference's own convf.c /
convi.c / gaussmat.c (oracle/_ref) and the properties the reference's
test_convolution.py pins.  GPU: the CUDA kernels against the oracle, bit-exact
(integer and float alike), through the C ABI."""
import numpy as np
import pytest

from oracle import pyconv, pyref
from oracle import pyoracle as orc
from refgold import ref  # noqa: F401

DTYPES = [np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32]

# test_convolution.py:43-55
SHARP = (np.array([[-1, -1, -1], [-1, 16, -1], [-1, -1, -1]], float), 8, 0)
BLUR = (np.array([[1, 1, 1], [1, 1, 1], [1, 1, 1]], float), 9, 0)
LINE = (np.array([[1, 1, 1], [-2, -2, -2], [1, 1, 1]], float), 1, 128)
SOBEL = (np.array([[1, 2, 1], [0, 0, 0], [-1, -2, -1]], float), 1, 128)
WIDE = (np.arange(35, dtype=float).reshape(5, 7) - 11.5, 3.5, -2.25)
MASKS = [SHARP, BLUR, LINE, SOBEL, WIDE]


def rnd(rng, dt, shape=(40, 50, 3)):
    dt = np.dtype(dt)
    if dt.kind == "f":
        return (rng.random(shape) * 255).astype(dt)
    i = np.iinfo(dt)
    return rng.integers(i.min, int(i.max) + 1, shape, dtype=np.int64).astype(dt)


def same(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype, (a.shape, b.shape, a.dtype, b.dtype)
    assert np.array_equal(a, b), "max diff %g" % np.abs(a.astype(np.float64) - b.astype(np.float64)).max()


# ------------------------------------------------------------------- CPU

def test_gaussmat_matches_reference(ref):
    for s, ma, sep, pr in ((0.5, 0.1, True, "integer"), (4.0, 0.2, True, "float"), (1.5, 0.2, False, "integer"),
                           (2.0, 0.2, False, "float"), (0.1, 0.2, True, "integer"), (7.3, 0.05, True, "float")):
        m1 = pyconv.gaussmat(s, ma, sep, pr)
        ref.check(m1[0], lambda: pyconv.ref_gaussmat(s, ma, sep, pr)[0])
        ref.check(np.array(m1[1:], np.float64), lambda: np.array(pyconv.ref_gaussmat(s, ma, sep, pr)[1:], np.float64))


def test_gaussmat_baseline_mask_is_15_taps():
    """SURVEY 8a10: sigma 4.0, min_ampl 0.2 => 15 taps; sharpen's sigma 0.5 / 0.1 => [3 20 3] / 26"""
    m, scale, _ = pyconv.gaussmat(4.0, 0.2, True, "float")
    assert m.shape == (1, 15)
    m, scale, _ = pyconv.gaussmat(0.5, 0.1, True, "integer")
    assert m.ravel().tolist() == [3, 20, 3] and scale == 26


@pytest.mark.parametrize("dt", DTYPES + [np.float64])
def test_oracle_conv_matches_reference(ref, dt):
    rng = np.random.default_rng(0)
    a = rnd(rng, dt)
    g15 = pyconv.gaussmat(4.0, 0.2, True, "float")
    for m, sc, off in MASKS + [(g15[0], g15[1], 0)]:
        for pr in ("float", "integer"):
            ref.check(pyconv.conv(a, m, sc, off, pr), lambda: pyconv.ref_conv(a, m, sc, off, pr))


def test_oracle_conv_vector_semantics_match_reference(ref):
    rng = np.random.default_rng(1)
    a = rnd(rng, np.uint8, (64, 64, 3))
    gi = pyconv.gaussmat(1.2, 0.2, False, "integer")
    for m, sc, off in MASKS + [(gi[0], gi[1], 0)]:
        ref.check(pyconv.conv(a, m, sc, off, "integer", vector=True), lambda: pyconv.ref_conv(a, m, sc, off, "integer", vector=True))


def test_conv_point_values():
    """test_convolution.py:68-86: conv == a direct point convolution at a pixel"""
    rng = np.random.default_rng(2)
    a = rnd(rng, np.uint8, (100, 100, 3))
    for m, sc, off in (SHARP, BLUR, LINE, SOBEL):
        f = pyconv.conv(a, m, sc, off, "float")
        for (x, y) in ((25, 50), (50, 50)):
            for b in range(3):
                want = off + (m * a[y - 1:y + 2, x - 1:x + 2, b].astype(float)).sum() / sc
                assert abs(f[y, x, b] - want) < 1e-3
                i = pyconv.conv(a, m, sc, off, "integer")[y, x, b]
                assert abs(int(i) - np.clip(want, 0, 255)) <= 1


def test_convsep_equals_conv_and_gaussblur():
    """test_convolution.py:138-157, 181-196"""
    rng = np.random.default_rng(3)
    a = rnd(rng, np.uint8, (60, 70, 3))
    m1, s1, _ = pyconv.gaussmat(2.0, 0.1, True, "float")
    m2, s2, _ = pyconv.gaussmat(2.0, 0.1, False, "float")
    sep = pyconv.convsep(a, m1, s1, 0, "float")
    full = pyconv.conv(a, m2, s2, 0, "float")
    assert np.abs(sep - full).max() < 0.1
    assert np.abs(pyconv.gaussblur(a, 2.0, 0.1, "float") - sep).max() == 0


def test_sharpen_identity_when_m1_m2_zero():
    """test_convolution.py:198-218: sharpen with m1 = m2 = 0 is the identity (max diff 0)"""
    rng = np.random.default_rng(4)
    a = rnd(rng, np.uint8, (50, 60, 3))
    for sigma in (0.5, 1, 1.5, 2):
        assert np.array_equal(pyconv.sharpen(a, "srgb", sigma=sigma, m1=0, m2=0), a)
    lab = orc.colourspace(a, "lab", "srgb")
    back = pyconv.sharpen(lab, "lab", m1=0, m2=0)
    assert np.abs(back - lab).max() < 0.01


def test_convsep_mask_orientation_against_reference(ref):
    """convsep.c:92-107 through the reference's own convsep.c / rot.c: an n x 1 mask runs the horizontal
    pass first; a 1 x n mask runs the vertical pass first and then the REVERSED row (vips_rot90), with
    the offset applied in the first pass only.  Asymmetric masks, integer rounding / clipping per pass."""
    rng = np.random.default_rng(21)
    row = np.array([[1.0, 4.0, 9.0, 2.0, -3.0]])
    for dt in (np.uint8, np.int16, np.float32):
        a = rnd(rng, dt, (40, 52, 3))
        for mask in (row, row.T.copy()):
            for pr in ("float", "integer"):
                got = pyconv.convsep(a, mask, 13.0, 7.0, pr)
                ref.check(got, lambda: pyconv.ref_convsep(a, mask, 13.0, 7.0, pr), (dt, mask.shape, pr))
    # and the orientation matters for these masks: the two orders differ
    assert not np.array_equal(pyconv.convsep(a, row, 13.0, 7.0, "integer"), pyconv.convsep(a, row.T.copy(), 13.0, 7.0, "integer"))


def test_sharpen_against_reference_sharpen_c(ref):
    """The reference's own sharpen.c (build: integer gaussmat at min_ampl 0.1, the LUT, L extraction,
    convsep; generate: sharpen.c:116-168) compiled into oracle/_ref: the oracle must equal it bit for
    bit -- LUT and pixels, several parameter sets, sRGB and LabS inputs, SMALLTILE and FATSTRIP sinks."""
    for kw in ({}, {"sigma": 1.5, "m2": 5.0, "y2": 20.0}, {"sigma": 0.8, "x1": 1.0, "m1": 0.5, "y3": 5.0}):
        lut_kw = {k: v for k, v in kw.items() if k != "sigma"}
        ref.check(pyconv.sharpen_lut(**lut_kw), lambda: pyconv.ref_sharpen_lut(**kw), kw)
    rng = np.random.default_rng(22)
    a = rnd(rng, np.uint8, (150, 170, 3))
    smooth = np.clip(np.add.outer(np.arange(150), np.arange(170))[:, :, None] * 0.7 + rng.integers(0, 12, (150, 170, 3)), 0, 255).astype(np.uint8)
    for img in (a, smooth):
        for kw in ({}, {"sigma": 1.5, "m2": 5.0, "y2": 20.0}, {"sigma": 0.8, "x1": 1.0, "m1": 0.5, "y3": 5.0}):
            got = pyconv.sharpen(img, "srgb", **kw)
            ref.check(got, lambda: pyconv.ref_sharpen(img, "srgb", **kw), kw)
            ref.check(got, lambda: pyconv.ref_sharpen(img, "srgb", tile=(128, 128), **kw), kw)  # tile-invariant
    labs = orc.colourspace(a, "labs", "srgb")
    ref.check(pyconv.sharpen(labs, "labs"), lambda: pyconv.ref_sharpen(labs, "labs"))


# ------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_gpu_conv(vb, dt):
    rng = np.random.default_rng(10)
    a = rnd(rng, dt, (61, 83, 3))
    g15 = pyconv.gaussmat(4.0, 0.2, True, "float")
    for m, sc, off in MASKS + [(g15[0], g15[1], 0)]:
        for pr in ("float", "integer"):
            same(vb.Image(a).conv(m, sc, off, pr).numpy(), pyconv.conv(a, m, sc, off, pr))


@pytest.mark.gpu
def test_gpu_conv_vector_semantics(vb):
    rng = np.random.default_rng(11)
    a = rnd(rng, np.uint8, (64, 96, 4))
    gi = pyconv.gaussmat(1.2, 0.2, False, "integer")
    try:
        vb.set_vector_convi(True)
        for m, sc, off in MASKS + [(gi[0], gi[1], 0)]:
            same(vb.Image(a).conv(m, sc, off, "integer").numpy(), pyconv.conv(a, m, sc, off, "integer", vector=True))
    finally:
        vb.set_vector_convi(False)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.uint8, np.uint16, np.int16, np.float32])
def test_gpu_convsep_gaussblur(vb, dt):
    rng = np.random.default_rng(12)
    a = rnd(rng, dt, (90, 70, 3))
    for pr in ("float", "integer"):
        m, sc, off = pyconv.gaussmat(4.0, 0.2, True, pr)
        same(vb.Image(a).convsep(m, sc, off, pr).numpy(), pyconv.convsep(a, m, sc, off, pr))
        for sigma in (0.1, 0.7, 2.5):
            same(vb.Image(a).gaussblur(sigma, 0.2, pr).numpy(), pyconv.gaussblur(a, sigma, 0.2, pr))
    g, s, o = vb.gaussmat(4.0, 0.2, True, "float")
    g2, s2, o2 = pyconv.gaussmat(4.0, 0.2, True, "float")
    assert np.array_equal(g, g2) and s == s2 and o == o2


@pytest.mark.gpu
def test_gpu_convsep_baseline_config3_reduced(vb):
    """BASELINE config 3 at reduced size: 15-tap float Gaussian on float RGB"""
    rng = np.random.default_rng(13)
    a = (rng.random((512, 768, 3)) * 255).astype(np.float32)
    m, sc, off = pyconv.gaussmat(4.0, 0.2, True, "float")
    same(vb.Image(a).convsep(m, sc, off, "float").numpy(), pyconv.convsep(a, m, sc, off, "float"))


@pytest.mark.gpu
def test_gpu_sharpen(vb):
    rng = np.random.default_rng(14)
    a = rnd(rng, np.uint8, (120, 150, 3))
    same(vb.Image(a, "srgb").sharpen().numpy(), pyconv.sharpen(a, "srgb"))
    same(vb.Image(a, "srgb").sharpen(sigma=1.5, m2=5.0, y2=20).numpy(), pyconv.sharpen(a, "srgb", sigma=1.5, m2=5.0, y2=20))
    rgba = rnd(rng, np.uint8, (64, 64, 4))
    same(vb.Image(rgba, "srgb").sharpen().numpy(), pyconv.sharpen(rgba, "srgb"))
    # identity when m1 = m2 = 0
    assert np.array_equal(vb.Image(a, "srgb").sharpen(m1=0, m2=0).numpy(), a)
    lab = orc.colourspace(a, "lab", "srgb")
    same(vb.Image(lab, "lab").sharpen().numpy(), pyconv.sharpen(lab, "lab"))


@pytest.mark.gpu
def test_gpu_convsep_mask_orientation(vb):
    rng = np.random.default_rng(23)
    row = np.array([[1.0, 4.0, 9.0, 2.0, -3.0]])
    for dt in (np.uint8, np.int16, np.float32):
        a = rnd(rng, dt, (40, 52, 3))
        for mask in (row, row.T.copy()):
            for pr in ("float", "integer"):
                same(vb.Image(a).convsep(mask, 13.0, 7.0, pr).numpy(), pyconv.convsep(a, mask, 13.0, 7.0, pr))
