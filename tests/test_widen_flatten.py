"""vips_flatten (SURVEY 8f rank 3).  CPU: the oracle against the reference's own conversion/flatten.c (+ cast.c) under
oracle/_ref over formats x bands x backgrounds x max_alpha settings, the kernel's per-pixel code compiled for the host
(vb200_debug_flatten_host, both the one-pixel and the four-pixel form) against the oracle, and the reference test-suite's
known answer.  GPU: the CUDA kernels against the oracle, bit for bit."""
import numpy as np
import pytest

from oracle import pyconv, pyref
from refgold import ref  # noqa: F401

DTYPES = (np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32)
sRGB, RGB16, scRGB = 22, 25, 28
SETTINGS = ((0, sRGB), (0, RGB16), (0, scRGB), (255, sRGB), (65535, sRGB), (1000, sRGB), (1, sRGB))


def image(rng, dt, shape):
    if np.dtype(dt).kind == "f":
        return (rng.random(shape) * 300 - 20).astype(dt)
    info = np.iinfo(dt)
    return rng.integers(max(info.min, -2 ** 31), min(info.max, 2 ** 32 - 1) + 1, shape, dtype=np.int64).astype(dt)


def backgrounds(bands):
    return ((0.0,), (10.7,), tuple(([300.2, -4, 77.9, 12.5, 1e6] * 4)[:bands - 1]), (0.0,) * (bands - 1))


def cases(rng, shapes):
    for dt in DTYPES:
        for shape in shapes:
            a = image(rng, dt, shape)
            for bg in backgrounds(shape[2]):
                for ma, interp in SETTINGS:
                    try:
                        want = pyconv.flatten(a, bg, ma, interp)
                    except NotImplementedError:
                        want = None  # the reference's arithmetic is undefined C there: the device path declines
                    yield a, bg, ma, interp, want


def test_oracle_flatten_matches_reference(ref):
    rng = np.random.default_rng(21)
    n = 0
    for a, bg, ma, interp, want in cases(rng, ((9, 13, 2), (7, 12, 4), (5, 6, 5))):
        if want is None:
            continue
        ref.check(want, lambda: pyconv.ref_flatten(a, bg, ma, interp), (a.dtype, a.shape, bg, ma, interp))
        n += 1
    assert n > 400
    a = image(rng, np.uint8, (40, 300, 4))
    ref.check(pyconv.flatten(a, (1, 2, 3)), lambda: pyconv.ref_flatten(a, (1, 2, 3), tile=(128, 16)))
    one = image(rng, np.uint16, (5, 5, 1))
    ref.check(one, lambda: pyconv.ref_flatten(one))
    assert np.array_equal(pyconv.flatten(one), one)


def test_host_twin_matches_oracle():
    import libvips_b200 as vb
    rng = np.random.default_rng(22)
    declined = 0
    for a, bg, ma, interp, want in cases(rng, ((9, 13, 2), (7, 12, 4), (5, 6, 5), (3, 5, 17))):
        if want is None:
            declined += 1
            with pytest.raises(vb.Error, match="not supported on the device path"):
                vb.flatten_host_twin(a, bg, ma, interp)
            continue
        got = vb.flatten_host_twin(a, bg, ma, interp)
        assert np.array_equal(got, want), (a.dtype, a.shape, bg, ma, interp)
        if a.dtype == np.uint8 and a.shape[2] == 4 and (ma or {sRGB: 255, RGB16: 65535, scRGB: 1}[interp]) >= 255:
            assert np.array_equal(vb.flatten_host_twin(a, bg, ma, interp, x4=True), want)
    assert declined > 0
    # every (value, alpha) pair through the uchar LUT paths, black and not
    v, al = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8))
    full = np.stack([v, v[::-1], v.T, al], axis=2)
    for bg in (None, (255, 0, 128.6)):
        want = pyconv.flatten(full, (0.0,) if bg is None else bg)
        assert np.array_equal(vb.flatten_host_twin(full, bg), want)
        assert np.array_equal(vb.flatten_host_twin(full, bg, x4=True), want)
    with pytest.raises(vb.Error, match="vector must have 1 or 3 elements"):
        vb.flatten_host_twin(full, (1, 2))
    with pytest.raises(vb.Error, match="bands not supported"):
        vb.flatten_host_twin(np.zeros((2, 2, 18), np.uint8))


def test_known_answers():
    """test/test-suite/test_conversion.py:369-413, restated on the oracle: (100, 128, 200 | alpha 127.5) cast to each
    format, flattened over black and over (100, 100, 100), lands within 2 of the arithmetic prediction; and an image whose
    max_alpha (255) is below its format's range clips the way the cast-at-the-end order says: flatten(ushort(rgba * 256))
    == ushort(flatten(float(rgba * 256)))"""
    import os
    for dt in (np.uint8, np.uint16, np.uint32, np.int16, np.int32, np.float32):
        px = np.empty((40, 40, 4), np.float64)
        px[:] = (100, 128, 200, 127.5)
        test = px.astype(dt)
        pixel = test[30, 30].astype(np.float64)
        mx, alpha = 255, 127.5
        nalpha = mx - alpha
        got = pyconv.flatten(test)
        assert got.shape == (40, 40, 3) and got.dtype == test.dtype
        for x, y in zip(got[30, 30], [int(v) * alpha / mx for v in pixel[:-1]]):
            assert abs(float(x) - y) < 2, (dt, x, y)
        got = pyconv.flatten(test, (100, 100, 100))
        for x, y in zip(got[30, 30], [int(v) * alpha / mx + 100 * nalpha / mx for v in pixel[:-1]]):
            assert abs(float(x) - y) < 2, (dt, x, y)
    rgba = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rgba_fixture.npz"))["rgba"]
    big = rgba.astype(np.float32) * 256
    im = pyconv.flatten(np.clip(big, 0, 65535).astype(np.uint16))           # rgba * 256, cast ushort, flatten
    im2 = np.clip(pyconv.flatten(big), 0, 65535).astype(np.uint16)          # rgba * 256, flatten, cast ushort
    assert np.array_equal(im, im2)


@pytest.mark.gpu
def test_gpu_flatten(vb):
    rng = np.random.default_rng(23)
    names = {sRGB: "srgb", RGB16: "rgb16", scRGB: "scrgb"}
    for a, bg, ma, interp, want in cases(rng, ((9, 13, 2), (37, 64, 4), (33, 41, 4), (5, 6, 5))):
        im = vb.Image(a, names[interp])
        if want is None:
            with pytest.raises(vb.Error, match="not supported on the device path"):
                im.flatten(bg, ma)
            continue
        got = im.flatten(bg, ma)
        assert got.array.dtype == want.dtype and np.array_equal(got.numpy(), want), (a.dtype, a.shape, bg, ma, interp)
    # the RGBA fast path at size, and all (value, alpha) pairs
    a = image(rng, np.uint8, (700, 1024, 4))
    assert np.array_equal(vb.Image(a).flatten((1, 2, 3)).numpy(), pyconv.flatten(a, (1, 2, 3)))
    assert np.array_equal(vb.Image(a).flatten().numpy(), pyconv.flatten(a))
    v, al = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8))
    full = np.stack([v, v[::-1], v.T, al], axis=2)
    assert np.array_equal(vb.Image(full).flatten((255, 0, 128.6)).numpy(), pyconv.flatten(full, (255, 0, 128.6)))
    one = image(rng, np.uint16, (5, 5, 1))
    assert np.array_equal(vb.Image(one).flatten().numpy(), one)
    # in a chain: flatten then median
    got = vb.Chain().flatten((9, 9, 9)).rank(3, 3, 4).run([a[:90, :120]])[0].numpy()
    assert np.array_equal(got, pyconv.median(pyconv.flatten(np.ascontiguousarray(a[:90, :120]), (9, 9, 9)), 3))
