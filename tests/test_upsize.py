"""Upsizing: vips_resize's affine half (resize.c:233-307) with the nearest /
bilinear / bicubic interpolators.  CPU: oracle against the reference's own
affine.c + interpolate.c + bicubic.cpp + resize.c; GPU: CUDA against the oracle."""
import numpy as np
import pytest

from oracle import pyoracle as orc
from oracle import pyref
from refgold import ref  # noqa: F401

DTYPES = [np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32]
CASES = [(2.0, None, "lanczos3"), (1.5, None, "cubic"), (1.3, 2.7, "linear"), (2.5, None, "nearest"),
         (3.1, 1.0, "lanczos3"), (1.0, 1.9, "mitchell"), (1.01, None, "linear")]


def rnd(rng, dt, shape=(40, 57, 3)):
    dt = np.dtype(dt)
    if dt.kind == "f":
        return (rng.random(shape) * 255).astype(dt)
    i = np.iinfo(dt)
    return rng.integers(i.min, int(i.max) + 1, shape, dtype=np.int64).astype(dt)


@pytest.mark.parametrize("dt", DTYPES)
def test_oracle_resize_up_matches_reference(ref, dt):
    rng = np.random.default_rng(1)
    a = rnd(rng, dt)
    for sc, vs, k in CASES:
        got = orc.resize(a, sc, vs, kernel=k)
        ref.check(got, lambda: pyref.RefImage.from_array(a).resize(sc, vs, kernel=k).numpy(), (sc, vs, k))


def test_resize_up_geometry_and_edges():
    a = np.full((10, 20, 3), 200, np.uint8)
    for k in ("nearest", "linear", "cubic", "lanczos3"):
        r = orc.resize(a, 2.5, kernel=k)
        assert r.shape == (25, 50, 3)
        assert (r == 200).all(), k  # constant image stays constant right up to the edges


def test_mixed_resize_is_rejected():
    a = np.zeros((20, 20, 1), np.uint8)
    with pytest.raises(ValueError):
        orc.resize(a, 2.0, 0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_gpu_resize_up(vb, dt):
    rng = np.random.default_rng(2)
    a = rnd(rng, dt, (61, 47, 4))
    for sc, vs, k in CASES:
        got = vb.Image(a).resize(sc, vs, kernel=k).numpy()
        want = orc.resize(a, sc, vs, kernel=k)
        assert got.shape == want.shape and np.array_equal(got, want), (sc, vs, k)


@pytest.mark.gpu
def test_gpu_thumbnail_up(vb):
    rng = np.random.default_rng(3)
    for bands in (3, 4):
        a = rng.integers(0, 256, (50, 80, bands), dtype=np.uint8)
        got = vb.Image(a).thumbnail_image(200).numpy()
        want = orc.thumbnail_image(a, 200)
        assert got.shape == want.shape == (125, 200, bands) and np.array_equal(got, want)


@pytest.mark.gpu
def test_gpu_mixed_and_zoom_fail_loudly(vb):
    a = np.zeros((20, 20, 1), np.uint8)
    with pytest.raises(vb.Error):
        vb.Image(a).resize(2.0, 0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.uint8, np.uint16, np.float32])
def test_gpu_zoom(vb, dt):
    """integral nearest enlargement is vips_zoom (resize.c:263-271): exact replication, also for factors
    like 3 and 7 where a coordinate built by repeated addition of 1 / scale would drift"""
    rng = np.random.default_rng(21)
    a = (rng.random((37, 53, 3)) * 200).astype(dt)
    for hs, vs in ((2.0, 2.0), (3.0, 7.0), (5.0, 1.0)):
        got = vb.Image(a).resize(hs, vs, kernel="nearest").numpy()
        want = np.repeat(np.repeat(a, int(vs), axis=0), int(hs), axis=1)
        assert np.array_equal(got, want)
        if vs > 1.0 or hs > 1.0:
            assert np.array_equal(orc.resize(a, hs, vs, kernel="nearest"), want)


@pytest.mark.gpu
@pytest.mark.parametrize("sc,vs", [(2.0, None), (3.7, 1.2), (1.0, 2.0), (1.25, 1.01), (4.0, 4.0)])
def test_gpu_separable_bicubic_rgba(vb, sc, vs):
    """the shared-memory separable form of the uchar RGBA bicubic upsize over many 64 x 32 tiles, ragged edges"""
    rng = np.random.default_rng(31)
    a = rnd(rng, np.uint8, (203, 317, 4))
    got = vb.Image(a).resize(sc, vs, kernel="cubic").numpy()
    want = orc.resize(a, sc, vs, kernel="cubic")
    assert got.shape == want.shape and np.array_equal(got, want)
