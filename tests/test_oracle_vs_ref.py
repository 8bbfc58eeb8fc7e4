"""CPU: pin the oracle restatement against the reference's OWN code.

oracle/_ref/libvipsref.so is the reference's resample/*.c*, conversion/*multiply.c,
colour/*.c and convolution/*.c compiled in place under a GLib-free shim (see
oracle/ref_shim/Makefile): its build() functions set up the ops, and a sink
pulls tiles through its generate() callbacks.  The restatement in oracle/*.cpp
must agree with it BIT FOR BIT, integer and float alike.

Where _ref has not been built, the reference's outputs come from the digests stored with the tests (tests/refgold.py).
"""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as orc
from oracle import pyref
from refgold import ref  # noqa: F401

DTYPES = [np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32, np.float64]
KERNELS = ["nearest", "linear", "cubic", "mitchell", "lanczos2", "lanczos3", "mks2013", "mks2021"]


def rand_image(rng, h, w, b, dt):
    dt = np.dtype(dt)
    if dt.kind == "f":
        return (rng.random((h, w, b)) * 255).astype(dt)
    info = np.iinfo(dt)
    return rng.integers(info.min, int(info.max) + 1, (h, w, b), dtype=np.int64).astype(dt)


@pytest.mark.parametrize("kernel", KERNELS)
def test_masks(ref, kernel):
    for shrink in (1.0, 1.1, 1.5, 2.0, 2.37, 8.0):
        n = orc.reduce_get_points(kernel, shrink)
        ref.check(n, lambda: pyref.reduce_get_points(kernel, shrink))
        for x in (0.0, 1 / 64.0, 0.5, 63 / 64.0, 1.0):
            ref.check(orc.reduce_make_mask(kernel, n, shrink, x), lambda: pyref.reduce_make_mask(kernel, n, shrink, x))


def test_mask_known_values():
    """SURVEY 8(c): shrink 2 => 13 taps, int mask sums to 4096; shrink 8 => 49 taps, 4090 / 4087"""
    _, s = orc.reduce_tables("lanczos3", 13, 2.0)
    assert s[0].tolist() == [15, 61, -139, -272, 555, 1828, 1828, 555, -272, -139, 61, 15, 0]
    _, s = orc.reduce_tables("lanczos3", 49, 8.0)
    assert s[0].sum() == 4090 and s[32].sum() == 4087


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("bands", [1, 3, 4])
def test_shrink(ref, dt, bands):
    rng = np.random.default_rng(2)
    a = rand_image(rng, 50, 71, bands, dt)
    r = lambda: pyref.RefImage.from_array(a)
    for f in (2, 3, 4, 5):
        for ceil in (False, True):
            ref.check(orc.shrinkv(a, f, ceil), lambda: r().shrinkv(f, ceil).numpy())
            ref.check(orc.shrinkh(a, f, ceil), lambda: r().shrinkh(f, ceil).numpy())


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("kernel", KERNELS)
def test_reduce(ref, dt, kernel):
    rng = np.random.default_rng(3)
    a = rand_image(rng, 45, 67, 3, dt)
    r = lambda: pyref.RefImage.from_array(a)
    for fac in (1.0, 1.1, 1.5, 1.999, 2.0, 3.3):
        # stand-alone reducev/reduceh are FATSTRIP ops: full-width x 16-row sink tiles
        ref.check(orc.reducev(a, fac, kernel, 0.0, rect_h=16), lambda: r().reducev(fac, kernel).numpy())
        ref.check(orc.reduceh(a, fac, kernel, 0.0, rect_w=0), lambda: r().reduceh(fac, kernel).numpy())


def test_reduce_tile_dependence_is_modelled(ref):
    """a shrink that is not exactly representable: the reference's result depends on
    the rect origin (Y += shrink per rect); the oracle's rect_h/rect_w reproduce it"""
    rng = np.random.default_rng(4)
    a = rand_image(rng, 400, 300, 1, np.uint8)
    r = lambda: pyref.RefImage.from_array(a)
    for th in (1, 7, 16, 128):
        ref.check(orc.reducev(a, 1.7, rect_h=th), lambda: r().reducev(1.7).numpy(tile=(300, th)))
    for tw in (1, 13, 64):
        ref.check(orc.reduceh(a, 1.7, rect_w=tw), lambda: r().reduceh(1.7).numpy(tile=(tw, 16)))


def test_reduce_gap(ref):
    rng = np.random.default_rng(5)
    a = rand_image(rng, 301, 257, 4, np.uint8)
    r = lambda: pyref.RefImage.from_array(a)

    def reducev(fac):
        rv = r().reducev(fac, gap=2.0)
        assert rv.dhint == 0  # SMALLTILE inherited from shrinkv
        return rv.numpy()
    for fac in (4.0, 5.5, 8.0, 9.4):
        ref.check(orc.reducev(a, fac, "lanczos3", 2.0, rect_h=128), lambda: reducev(fac))
        ref.check(orc.reduceh(a, fac, "lanczos3", 2.0, rect_w=0), lambda: r().reduceh(fac, gap=2.0).numpy())


@pytest.mark.parametrize("dt", DTYPES)
def test_premultiply(ref, dt):
    rng = np.random.default_rng(6)
    for bands in (2, 4, 5):
        a = rand_image(rng, 21, 33, bands, dt)
        r = lambda: pyref.RefImage.from_array(a)
        ref.check(orc.premultiply(a, 255.0, False), lambda: r().premultiply(255.0).numpy())
        if bands == 4:
            ref.check(orc.unpremultiply(a, 255.0, False), lambda: r().unpremultiply(255.0).numpy())
        if dt == np.uint8:
            ref.check(orc.premultiply(a, 255.0, True), lambda: r().premultiply(uchar=True).numpy())
            if bands == 4:
                ref.check(orc.unpremultiply(a, 255.0, True), lambda: r().unpremultiply(uchar=True).numpy())


def test_premultiply_all_alpha_values(ref):
    v, al = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8))
    a = np.ascontiguousarray(np.stack([v, v[::-1], v.T, al], axis=-1))
    r = lambda: pyref.RefImage.from_array(a)
    ref.check(orc.premultiply(a, 255.0, True), lambda: r().premultiply(uchar=True).numpy())
    ref.check(orc.unpremultiply(a, 255.0, True), lambda: r().unpremultiply(uchar=True).numpy())


@pytest.mark.parametrize("dt", [np.uint8, np.uint16, np.int16, np.float32])
def test_resize(ref, dt):
    rng = np.random.default_rng(7)
    a = rand_image(rng, 300, 401, 3, dt)
    r = lambda: pyref.RefImage.from_array(a)
    for scale in (0.25, 0.5, 0.37, 0.13, 0.9, 0.111):
        ref.check(orc.resize(a, scale), lambda: r().resize(scale).numpy())
    ref.check(orc.resize(a, 0.3, 0.7, kernel="cubic"), lambda: r().resize(0.3, 0.7, kernel="cubic").numpy())
    ref.check(orc.resize(a, 0.3, 0.7, kernel="linear", gap=0.0), lambda: r().resize(0.3, 0.7, kernel="linear", gap=0.0).numpy())


@pytest.mark.parametrize("shape,target", [((1024, 1024), 128), ((997, 761), 100), ((640, 480), 64),
                                           ((300, 300), 150), ((333, 1999), 77), ((2048, 1024), 300)])
@pytest.mark.parametrize("bands", [3, 4])
def test_thumbnail_chain(ref, shape, target, bands):
    rng = np.random.default_rng(8)
    a = rng.integers(0, 256, shape + (bands,), dtype=np.uint8)
    ref.check(orc.thumbnail_image(a, target), lambda: pyref.thumbnail_image(a, target))


def test_thumbnail_size_arithmetic(ref):
    """vips_thumbnail_calculate_shrink / _find_jpegshrink (thumbnail.c:412-517), the file-static functions themselves
    (ref_shim/ref_thumbnail.c), against the oracle's restatement and the library's host-side rule"""
    import libvips_b200 as vb
    rng = np.random.default_rng(21)
    dims = [(4096, 4096), (6000, 4000), (4000, 6000), (800, 600), (1, 1), (1, 5000), (5000, 1), (997, 761), (65535, 3), (33, 32)]
    dims += [tuple(int(v) for v in rng.integers(1, 9000, 2)) for _ in range(300)]
    targets = [(512, None), (1, None), (7, 9000), (9000, 7), (300, 300), (1024, 1025), (100000, 2)]
    targets += [tuple(int(v) for v in rng.integers(1, 5000, 2)) for _ in range(40)]
    calls = [(w, h, tw, th, size) for (w, h) in dims for (tw, th) in targets for size in ("both", "up", "down", "force")]
    assert len(calls) > 50000
    shrinks, jpegshrinks = [], []
    for (w, h, tw, th, size) in calls:
        # the shrinks are written before the resize geometry is worked out (which declines mixed up / down sizes)
        ohs, ovs, ow, oh = C.c_double(), C.c_double(), C.c_int(), C.c_int()
        orc.lib().orc_thumbnail_size(w, h, tw, tw if th is None else th, orc.SIZES[size], C.byref(ohs), C.byref(ovs),
                                     C.byref(ow), C.byref(oh))
        shrinks.append((ohs.value, ovs.value))
        jpegshrinks.append(vb.thumbnail_jpegshrink(w, h, tw, th, size))
    ref.check(np.array(shrinks), lambda: np.array([pyref.thumbnail_calculate_shrink(*c) for c in calls]))
    ref.check(np.array(jpegshrinks), lambda: np.array([pyref.thumbnail_find_jpegshrink(*c) for c in calls]))
    ref.check(np.ones(len(calls), int), lambda: np.array([pyref.thumbnail_find_jpegshrink(*c, linear=True) for c in calls]))


def test_thumbnail_chain_tile_geometries(ref):
    rng = np.random.default_rng(9)
    a = rng.integers(0, 256, (999, 1001, 4), dtype=np.uint8)
    for tile in ((64, 64), (128, 128), (10, 10)):
        ref.check(orc.thumbnail_image(a, 123, tile=tile), lambda: pyref.thumbnail_image(a, 123, tile=tile))
