"""The B_W / GREY16 / HSV rows of vips_colourspace (SURVEY 8f rank 3, second lot).

CPU: the oracle's restatements of sRGB2HSV.c / HSV2sRGB.c (every one of the 2^24 inputs, both ways) and scRGB2BW.c against
the reference's own line functions under oracle/_ref; the whole of vips_colourspace for every pair that touches the three
spaces -- colourspace.c's route table, BW2sRGB / GREY162RGB16 (vips__colourspace_process_n over bandjoin), a real
VipsColour object per converter with its alpha handling -- against the oracle; the product's host twins of the new
per-pixel arithmetic against the oracle.  GPU: the CUDA path against the oracle, bit for bit (uchar / ushort results)
or exactly equal floats (the float steps of these routes are the existing, exact ones)."""
import numpy as np
import pytest

from oracle import pyoracle as orc
from oracle import pyref
from refgold import ref  # noqa: F401

TRUNK = ["srgb", "scrgb", "xyz", "lab", "labs", "rgb16", "lch", "yxy"]
EXT = ["b-w", "grey16", "hsv"]


def all_triples():
    v = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], axis=1).astype(np.uint8)


def sample(space, rng, n, bands):
    """n pixels of `bands` bands in the space's own format: the colour bands first, then extra bands"""
    main = 1 if space in ("b-w", "grey16") else 3
    if space in ("srgb", "hsv", "b-w"):
        a = rng.integers(0, 256, (n, bands), dtype=np.uint8)
    elif space in ("rgb16", "grey16"):
        a = rng.integers(0, 65536, (n, bands), dtype=np.uint16)
    elif space == "labs":
        a = rng.integers(-32768, 32768, (n, bands), dtype=np.int64).astype(np.int16)
        a[:, 0] = np.abs(a[:, 0])
    elif space == "scrgb":
        a = rng.random((n, bands), dtype=np.float32) * 1.2 - 0.1
    elif space == "xyz":
        a = rng.random((n, bands), dtype=np.float32) * 110 - 5
    elif space == "lch":
        a = rng.random((n, bands), dtype=np.float32) * np.array(([100, 130, 360] + [255] * 8)[:bands], np.float32)
    elif space == "yxy":
        a = rng.random((n, bands), dtype=np.float32) * np.array(([100, 1, 1] + [255] * 8)[:bands], np.float32)
    else:
        a = rng.random((n, bands), dtype=np.float32)
        a[:, 0] *= 100
        a[:, 1:3] = a[:, 1:3] * 256 - 128
        a[:, 3:] *= 255
    assert bands >= main
    return a


def pairs():
    for src in TRUNK + EXT:
        for dst in TRUNK + EXT:
            if src in EXT or dst in EXT:
                yield src, dst


def test_oracle_hsv_lines_match_reference_on_every_input(ref):
    a = all_triples()
    for step in ("sRGB2HSV", "HSV2sRGB"):
        got = orc.colour_step(a.reshape(4096, 4096, 3), step, "srgb" if step == "sRGB2HSV" else "hsv").reshape(-1, 3)
        ref.check(got, lambda: pyref.colour_line(step, a), step)


@pytest.mark.parametrize("step", ["scRGB2BW", "scRGB2BW16"])
def test_oracle_bw_line_matches_reference(ref, step):
    rng = np.random.default_rng(51)
    a = rng.random((200000, 3), dtype=np.float32) * 1.3 - 0.15
    a[::97, 0] = np.nan
    a[::89, 1] = np.inf
    a[::83, 2] = -np.inf
    a[::7] = np.round(a[::7] * 255) / 255  # exact table knots
    got = orc.colour_step(a.reshape(1, -1, 3), step, "scrgb").reshape(-1, 1)
    ref.check(got, lambda: pyref.colour_line(step, a))


def test_routes_follow_the_table():
    """colourspace.c:223-497, spot rows spelled out"""
    import ctypes as C
    steps = (C.c_int * 8)()
    name = {v: k for k, v in orc.STEPS.items()}
    rows = {("srgb", "b-w"): ["sRGB2scRGB", "scRGB2BW"], ("b-w", "srgb"): ["BW2sRGB"], ("b-w", "lab"): ["BW2sRGB", "sRGB2scRGB", "scRGB2XYZ", "XYZ2Lab"],
            ("grey16", "srgb"): ["GREY162RGB16", "RGB162sRGB"], ("grey16", "b-w"): ["GREY162RGB16", "RGB162scRGB", "scRGB2BW"],
            ("b-w", "grey16"): ["BW2sRGB", "sRGB2scRGB", "scRGB2BW16"], ("lab", "hsv"): ["Lab2XYZ", "XYZ2scRGB", "scRGB2sRGB", "sRGB2HSV"],
            ("hsv", "lch"): ["HSV2sRGB", "sRGB2scRGB", "scRGB2XYZ", "XYZ2Lab", "Lab2LCh"], ("rgb16", "hsv"): ["RGB162sRGB", "sRGB2HSV"],
            ("hsv", "rgb16"): ["HSV2sRGB", "sRGB2RGB16"], ("lch", "b-w"): ["LCh2Lab", "Lab2XYZ", "XYZ2scRGB", "scRGB2BW"],
            ("yxy", "grey16"): ["Yxy2XYZ", "XYZ2scRGB", "scRGB2BW16"], ("b-w", "hsv"): ["BW2sRGB", "sRGB2HSV"], ("hsv", "b-w"): ["HSV2sRGB", "sRGB2scRGB", "scRGB2BW"]}
    for (a, b), want in rows.items():
        n = orc.lib().orc_colourspace_route(orc.SPACES[a], orc.SPACES[b], steps)
        assert [name[steps[i]] for i in range(n)] == want, (a, b)


@pytest.mark.parametrize("extra", [0, 1, 2])
def test_oracle_colourspace_matches_reference_build(ref, extra):
    rng = np.random.default_rng(60 + extra)
    for src, dst in pairs():
        bands = (1 if src in ("b-w", "grey16") else 3) + extra
        a = sample(src, rng, 31 * 47, bands).reshape(31, 47, bands)
        got = orc.colourspace(a, dst, src)
        ref.check(got, lambda: pyref.RefImage.from_array(a, orc.SPACES[src]).colourspace(dst, src).numpy(tile=(16, 8)), (src, dst, extra))


def test_oracle_colourspace_foreign_formats_match_reference_build(ref):
    """images whose format is not the one the interpretation implies: the converters cast the whole image first; B_W ->
    sRGB and GREY16 -> RGB16 alone keep whatever format came in (a bandjoin)"""
    rng = np.random.default_rng(71)
    for dt in (np.uint8, np.uint16, np.int16, np.float32):
        for src, dst in pairs():
            bands = (1 if src in ("b-w", "grey16") else 3) + 1
            if dt == np.float32:
                a = (rng.standard_normal((13, 17, bands)) * 200).astype(np.float32)
            else:
                a = rng.integers(np.iinfo(dt).min, np.iinfo(dt).max + 1, (13, 17, bands)).astype(dt)
            try:
                got = orc.colourspace(a, dst, src)
            except ValueError:
                # the shifting casts from a format that is neither uchar nor ushort are not restated (tests/test_colour.py)
                assert dt not in (np.uint8, np.uint16), (dt, src, dst)
                continue
            ref.check(got, lambda: pyref.RefImage.from_array(a, orc.SPACES[src]).colourspace(dst, src).numpy(), (dt, src, dst))


def test_hsv_host_twin_matches_oracle_on_every_input():
    """hsv_kernel's per-pixel code (explicit round-to-nearest operations, fmodf(x, 2) as x - 2 floor(x / 2)) compiled
    for the host, against the oracle (which the test above pins to the reference): all 2^24 inputs, both ways"""
    import libvips_b200 as vb
    a = all_triples()
    for step, to_hsv in (("sRGB2HSV", True), ("HSV2sRGB", False)):
        want = orc.colour_step(a.reshape(4096, 4096, 3), step, "srgb" if to_hsv else "hsv").reshape(-1, 3)
        assert np.array_equal(vb.hsv_host_twin(a, to_hsv), want), step


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [0, 1])
def test_gpu_routes(vb, extra):
    rng = np.random.default_rng(80 + extra)
    for src, dst in pairs():
        if "lch" in (src, dst):
            continue  # the two LCh steps call atan / cosf / sinf (1 ULP against glibc): tests/test_colour.py holds them
        bands = (1 if src in ("b-w", "grey16") else 3) + extra
        a = sample(src, rng, 67 * 129, bands).reshape(67, 129, bands)
        got = vb.Image(a, src).colourspace(dst)
        want = orc.colourspace(a, dst, src)
        assert got.array.dtype == want.dtype and got.array.shape == want.shape, (src, dst)
        assert np.array_equal(got.numpy(), want, equal_nan=True), (src, dst, extra)
        assert got.interpretation == vb.INTERPRETATIONS[dst]


@pytest.mark.gpu
def test_gpu_hsv_every_input_and_greyscale_at_size(vb):
    a = all_triples().reshape(4096, 4096, 3)
    hsv = vb.Image(a, "srgb").colourspace("hsv").numpy()
    assert np.array_equal(hsv, orc.colour_step(a, "sRGB2HSV", "srgb"))
    assert np.array_equal(vb.Image(a, "hsv").colourspace("srgb").numpy(), orc.colour_step(a, "HSV2sRGB", "hsv"))
    # the common call: sRGB -> B_W, one launch, every sRGB triple
    before = vb.launch_count()
    bw = vb.Image(a, "srgb").colourspace("b-w").numpy()
    assert vb.launch_count() - before == 1
    assert bw.shape == (4096, 4096, 1) and np.array_equal(bw, orc.colourspace(a, "b-w", "srgb"))
    # grey -> rgb -> grey is the identity (8 and 16 bit)
    g = np.arange(256, dtype=np.uint8).reshape(16, 16, 1)
    assert np.array_equal(vb.Image(g, "b-w").colourspace("srgb").colourspace("b-w").numpy(), g)
    with pytest.raises(vb.Error, match="wants band format"):
        vb.Image(g.astype(np.float32), "b-w").colourspace("srgb")
    # in a chain: greyscale, then a median
    from oracle import pyconv
    c = np.ascontiguousarray(a[:90, :120])
    got = vb.Chain().colourspace("b-w").rank(3, 3, 4).run([c])[0].numpy()
    assert np.array_equal(got, pyconv.median(orc.colourspace(c, "b-w", "srgb"), 3))


def test_known_answer_grey_colour_grey():
    """test/test-suite/test_colour.py:59-74: Lab (50, 0, 0) + alpha 42 to a mono space, from there through every colour
    space in turn and back to the mono space: the 8-bit grey comes back exactly, the 16-bit one within 30, alpha within 1
    (the reference's list also holds CMC and the Oklab pair, which are not built here)"""
    test = np.empty((20, 20, 4), np.float32)
    test[:] = (50, 0, 0, 42)
    for mono, bound in (("b-w", 1), ("grey16", 30)):
        grey = orc.colourspace(test, mono, "lab")
        assert grey.shape == (20, 20, 2)
        im, space = grey, mono
        for col in ("xyz", "lab", "lch", "labs", "scrgb", "hsv", "srgb", "yxy", mono):
            im = orc.colourspace(im, col, space)
            space = col
        assert im.shape == grey.shape and im.dtype == grey.dtype
        assert abs(int(im[10, 10, 0]) - int(grey[10, 10, 0])) < bound, (mono, im[10, 10], grey[10, 10])
        assert abs(int(im[10, 10, 1]) - int(grey[10, 10, 1])) < 1, (mono, im[10, 10], grey[10, 10])


def test_oracle_colourspace_wild_floats_match_reference_build(ref):
    """NaN / Inf pixels and NaN alpha into the three spaces: scRGB2BW throws NaN luminance out (LabQ2sRGB.c:405-409), the clip
    handles the infinities, the alpha cast is the reference's own"""
    rng = np.random.default_rng(9)
    for bands in (3, 4):
        for src in ("scrgb", "xyz", "lab", "lch", "yxy"):
            a = (rng.standard_normal((23, 40, bands)) * 150).astype(np.float32)
            a[::7, ::5, 0] = np.nan
            a[::5, ::3, 1] = np.inf
            a[::3, ::7, 2] = -np.inf
            if bands == 4:
                a[::2, ::2, 3] = np.nan
            for dst in EXT:
                got = orc.colourspace(a, dst, src)
                ref.check(got, lambda: pyref.RefImage.from_array(a, orc.SPACES[src]).colourspace(dst, src).numpy(), (src, dst, bands))
