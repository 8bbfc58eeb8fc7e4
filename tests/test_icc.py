"""ICC rows (SURVEY 8a a20): vb200_icc_import / _export / _transform.

The reference's arithmetic is inside lcms2 (icc_transform.c:459, :931, :1094, :1219), which pins
no version; oracle/pylcms.py binds the lcms2 2.18 that ships with Pillow and makes the reference's
exact calls.  The CUDA path is a from-specification ICC evaluator: parity is a TOLERANCE against
lcms2 (its 8 / 16-bit transforms are table interpolations of the same colorimetry), stated per case
below and far inside the reference's own bounds (test_colour.py:128-178: dE76 < 6, |diff| < 3).

CPU tests run the evaluator's own per-pixel code on the host (vb200_debug_icc_eval, the same
__host__ __device__ functions the kernel calls); GPU tests require the kernel to agree with that."""
import ctypes as C
import os

import numpy as np
import pytest

import icc_fixtures as F
import libvips_b200 as vb
from oracle import pylcms

needs_lcms = pytest.mark.skipif(not pylcms.available(), reason="no lcms2 next to Pillow")
FMT = {np.dtype(np.uint8): 0, np.dtype(np.uint16): 2, np.dtype(np.float32): 6}
# the reference's own profiles (libvips/colour/profiles), copied by tests/golden/make_ref_profiles.py
REF_PROFILES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "profiles")


def host_eval(mode, a, pa, pb=None, depth=8, pcs=0, intent=1):
    L = C.CDLL(vb.library_path())
    L.vb200_debug_icc_eval.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_size_t,
                                       C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_int]
    L.vb200_error_buffer.restype = C.c_char_p
    a = np.ascontiguousarray(a)
    n = a.size // a.shape[-1]
    out = np.zeros((n, 8), np.float32 if mode == 0 else (np.uint8 if depth == 8 else np.uint16))
    ob = L.vb200_debug_icc_eval(mode, a.ctypes.data, FMT[a.dtype], a.shape[-1], out.ctypes.data, n, pa, len(pa), pb,
                                len(pb) if pb else 0, intent, depth, pcs)
    if ob < 0:
        raise vb.Error(L.vb200_error_buffer().decode(errors="replace"))
    return np.ascontiguousarray(out.reshape(-1)[: n * ob].reshape(n, ob))


def de(a, b):
    return np.sqrt(((a.astype(np.float64) - b) ** 2).sum(axis=-1))


@needs_lcms
@pytest.mark.parametrize("trc", ["srgb", "gamma", "para4", "table"])
def test_matrix_profiles_against_lcms2(trc):
    prof = F.rgb_profile(trc)
    rng = np.random.default_rng(3)
    a8 = rng.integers(0, 256, (40000, 3), dtype=np.uint8)
    lab = pylcms.icc_import(a8, prof)
    # 8-bit import: lcms2 interpolates a prelinearised 33-point CLUT; we evaluate the curves and the matrix
    # (a steep table TRC is where its interpolation is coarsest: dark colours, dE up to ~1.4)
    assert de(host_eval(0, a8, prof), lab).max() < {"table": 1.6}.get(trc, 0.8)
    assert de(host_eval(0, a8, prof), lab).mean() < 0.05
    # float import: lcms2 evaluates its float pipeline: agreement to the Lab16 quantum
    af = rng.random((40000, 3), dtype=np.float32)
    assert np.abs(host_eval(0, af, prof) - pylcms.icc_import(af, prof)).max() < 0.03
    # export from Lab float is lcms2's float pipeline too: at most 1 LSB, almost always 0
    d = np.abs(host_eval(1, lab, prof).astype(int) - pylcms.icc_export(lab, prof).astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.002
    d = np.abs(host_eval(1, lab, prof, depth=16).astype(int) - pylcms.icc_export(lab, prof, depth=16).astype(int))
    assert d.max() <= 128 and d.mean() < 2               # a table TRC is inverted by search here, by a reversed 4096-point table there
    # XYZ PCS (decode_xyz / encode_xyz with the reference's Bradford matrices)
    assert np.abs(host_eval(0, a8, prof, pcs=1) - pylcms.icc_import(a8, prof, pcs="xyz")).max() < 0.08
    xyz = pylcms.icc_import(a8, prof, pcs="xyz")
    d = np.abs(host_eval(1, xyz, prof, pcs=1).astype(int) - pylcms.icc_export(xyz, prof, pcs="xyz").astype(int))
    assert d.max() <= 1


@needs_lcms
@pytest.mark.parametrize("intent", ["perceptual", "saturation"])
def test_matrix_profiles_other_intents(intent):
    """lcms2 turns black point compensation on for these intents against the v4 PCS profiles; for a matrix or grey
    profile whose black is XYZ 0 that is the identity, and lcms2's own output is bit-identical to its relative one"""
    prof, code = F.rgb_profile("srgb"), {"perceptual": 0, "saturation": 2}[intent]
    a = np.random.default_rng(13).integers(0, 256, (20000, 3), dtype=np.uint8)
    assert np.array_equal(pylcms.icc_import(a, prof, intent), pylcms.icc_import(a, prof, "relative"))
    assert np.array_equal(host_eval(0, a, prof, intent=code), host_eval(0, a, prof))
    lab = pylcms.icc_import(a, prof)
    assert np.array_equal(pylcms.icc_export(lab, prof, intent), pylcms.icc_export(lab, prof, "relative"))
    assert np.array_equal(host_eval(1, lab, prof, intent=code), host_eval(1, lab, prof))
    g = np.arange(256, dtype=np.uint8).reshape(-1, 1)
    assert np.array_equal(pylcms.icc_import(g, F.grey_profile(), intent), pylcms.icc_import(g, F.grey_profile(), "relative"))


def _rgb_profile_with_white(white, version=0x04200000, cls="mntr", trc="srgb"):
    curve = F._para(*F._SRGB_PARA) if trc == "srgb" else F._curv([2.2])
    tags = [("desc", F._text("desc", "vb200 test rgb")), ("cprt", F._text("cprt", "none")), ("wtpt", F._xyz_tag(*white))]
    for name, col in zip("rgb", F._SRGB_COL):
        tags.append((name + "XYZ", F._xyz_tag(*col)))
    for name in "rgb":
        tags.append((name + "TRC", curve))
    return F._profile(version, cls, "RGB ", "XYZ ", tags)


@needs_lcms
@pytest.mark.parametrize("white", [(0.90, 1.0, 0.70), (0.9642, 1.0, 0.8249), (0.95, 0.98, 1.05)])
@pytest.mark.parametrize("version,cls", [(0x04200000, "mntr"), (0x02100000, "mntr"), (0x02100000, "scnr")])
def test_absolute_colorimetric_against_lcms2(white, version, cls):
    """intent 3 on matrix / TRC profiles: the relative transform with PCS XYZ scaled by media white over the other end's
    media white (lcms2 ComputeAbsoluteIntent, adaptation state 1): the wtpt tag, but D50 for a v2 display profile; D50 for
    the XYZ PCS profile; the D65 white of cmsWhitePointFromTemp(6504) for the reference's Lab PCS profile -- so with the
    default Lab PCS even a D50 profile is scaled.  Same tolerances as the relative intent."""
    prof = _rgb_profile_with_white(white, version, cls)
    rng = np.random.default_rng(13)
    a8 = rng.integers(0, 256, (20000, 3), dtype=np.uint8)
    lab = pylcms.icc_import(a8, prof, "absolute")
    assert de(lab, pylcms.icc_import(a8, prof, "relative")).max() > 2      # it is another transform
    d = de(host_eval(0, a8, prof, intent=3), lab)
    assert d.max() < 0.8 and d.mean() < 0.05
    af = rng.random((20000, 3), dtype=np.float32)
    assert np.abs(host_eval(0, af, prof, intent=3) - pylcms.icc_import(af, prof, "absolute")).max() < 0.03
    d = np.abs(host_eval(1, lab, prof, intent=3).astype(int) - pylcms.icc_export(lab, prof, "absolute").astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.002
    xyz = pylcms.icc_import(a8, prof, "absolute", pcs="xyz")
    assert np.abs(host_eval(0, a8, prof, pcs=1, intent=3) - xyz).max() < 0.08
    d = np.abs(host_eval(1, xyz, prof, pcs=1, intent=3).astype(int) - pylcms.icc_export(xyz, prof, "absolute", pcs="xyz").astype(int))
    assert d.max() <= 1
    # device to device: the two media whites against each other.  lcms2 evaluates float input exactly and resamples 8-bit
    # input into a CLUT (the scale stage defeats its matrix-shaper shortcut): hold the first to 1 / 65535, the second as colours
    other = _rgb_profile_with_white((0.95, 0.98, 1.05), 0x02100000, "scnr", "gamma")
    f = (a8 / 255.0).astype(np.float32)
    d = np.abs(host_eval(2, f, prof, other, intent=3, depth=16).astype(int) - pylcms.icc_transform(f, prof, other, "absolute", depth=16).astype(int))
    assert d.max() <= 2 and d.mean() < 0.01
    ours, theirs = host_eval(2, a8, prof, other, intent=3), pylcms.icc_transform(a8, prof, other, "absolute")
    d = de(pylcms.icc_import(ours, other), pylcms.icc_import(theirs, other))
    # the differences sit where the scaled colour leaves the target gamut and lcms2's 33-point CLUT interpolates across the clip
    assert d.max() < 6.0 and np.percentile(d, 99) < 3.0 and d.mean() < 0.2, (d.max(), np.percentile(d, 99), d.mean())


@needs_lcms
def test_rgb_to_rgb_transform_against_lcms2():
    pa, pb = F.rgb_profile("srgb"), F.rgb_profile("gamma")
    a = np.random.default_rng(4).integers(0, 256, (40000, 3), dtype=np.uint8)
    d = np.abs(host_eval(2, a, pa, pb).astype(int) - pylcms.icc_transform(a, pa, pb).astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.03     # lcms2 runs this one in 1.14 fixed point
    a16 = np.random.default_rng(5).integers(0, 65536, (40000, 3), dtype=np.uint16)
    d = np.abs(host_eval(2, a16, pa, pb, depth=16).astype(int) - pylcms.icc_transform(a16, pa, pb, depth=16).astype(int))
    assert d.max() <= 256 and d.mean() < 6            # <= 1 LSB of 8 bits


@needs_lcms
def test_grey_profile_against_lcms2():
    prof = F.grey_profile()
    g = np.arange(256, dtype=np.uint8).reshape(-1, 1)
    lab = pylcms.icc_import(g, prof)
    assert de(host_eval(0, g, prof), lab).max() < 0.3
    assert np.array_equal(host_eval(1, lab, prof), pylcms.icc_export(lab, prof))


@needs_lcms
def test_lut_profile_against_lcms2():
    ink, rgb = F.ink_profile(), F.rgb_profile()
    rng = np.random.default_rng(6)
    c = rng.integers(0, 256, (40000, 4), dtype=np.uint8)
    # A2B: 4-input lut16, tetrahedral over 3 + linear over the first channel, like lcms2's Eval4Inputs
    assert de(host_eval(0, c, ink), pylcms.icc_import(c, ink)).max() < 1.5
    lab = pylcms.icc_import(rng.integers(0, 256, (40000, 3), dtype=np.uint8), rgb)
    # B2A of a Lab-PCS profile: trilinear, like lcms2
    d = np.abs(host_eval(1, lab, ink).astype(int) - pylcms.icc_export(lab, ink).astype(int))
    assert d.max() <= 2 and d.mean() < 0.05
    # device to device: compare the COLOURS of the two ink answers (lcms2 precomputes a CLUT of the chain)
    a = rng.integers(0, 256, (40000, 3), dtype=np.uint8)
    ours, theirs = host_eval(2, a, rgb, ink), pylcms.icc_transform(a, rgb, ink)
    assert de(pylcms.icc_import(ours, ink), pylcms.icc_import(theirs, ink)).max() < 3.0
    d = np.abs(host_eval(2, c, ink, rgb).astype(int) - pylcms.icc_transform(c, ink, rgb).astype(int))
    assert d.mean() < 1.0 and np.percentile(d, 99) <= 3


@needs_lcms
@pytest.mark.parametrize("pcs", ["XYZ ", "Lab "])
def test_v4_lut_profile_against_lcms2(pcs):
    """lutAtoB / lutBtoA tags (A curves, CLUT on a non-uniform grid, M curves, matrix, B curves)"""
    prof, rgb = F.lut_v4_rgb_profile(pcs), F.rgb_profile()
    rng = np.random.default_rng(12)
    a = rng.integers(0, 256, (30000, 3), dtype=np.uint8)
    af = rng.random((30000, 3), dtype=np.float32)
    assert de(host_eval(0, a, prof), pylcms.icc_import(a, prof)).max() < 1.6
    assert np.abs(host_eval(0, af, prof) - pylcms.icc_import(af, prof)).max() < 0.04
    lab = pylcms.icc_import(a, rgb)
    d = np.abs(host_eval(1, lab, prof).astype(int) - pylcms.icc_export(lab, prof).astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.005
    d = np.abs(host_eval(2, a, prof, rgb).astype(int) - pylcms.icc_transform(a, prof, rgb).astype(int))
    assert d.max() <= 5 and d.mean() < 0.2
    d = np.abs(host_eval(2, a, rgb, prof).astype(int) - pylcms.icc_transform(a, rgb, prof).astype(int))
    assert d.max() <= 10 and d.mean() < 0.3


@needs_lcms
def test_reference_profiles_against_lcms2():
    P = lambda n: open(os.path.join(REF_PROFILES, n), "rb").read()
    rng = np.random.default_rng(7)
    a = rng.integers(0, 256, (30000, 3), dtype=np.uint8)
    for name in ("sRGB.icm", "p3.icm"):
        lab = pylcms.icc_import(a, P(name))
        assert de(host_eval(0, a, P(name)), lab).max() < 0.8
        d = np.abs(host_eval(1, lab, P(name)).astype(int) - pylcms.icc_export(lab, P(name)).astype(int))
        assert d.max() <= 1 and (d > 0).mean() < 0.002
    d = np.abs(host_eval(2, a, P("sRGB.icm"), P("p3.icm")).astype(int) - pylcms.icc_transform(a, P("sRGB.icm"), P("p3.icm")).astype(int))
    assert d.max() <= 1
    c = rng.integers(0, 256, (30000, 4), dtype=np.uint8)
    assert de(host_eval(0, c, P("cmyk.icm")), pylcms.icc_import(c, P("cmyk.icm"))).max() < 1.5
    lab = pylcms.icc_import(a, P("sRGB.icm"))
    d = np.abs(host_eval(1, lab, P("cmyk.icm")).astype(int) - pylcms.icc_export(lab, P("cmyk.icm")).astype(int))
    assert d.max() <= 1
    ours, theirs = host_eval(2, a, P("sRGB.icm"), P("cmyk.icm")), pylcms.icc_transform(a, P("sRGB.icm"), P("cmyk.icm"))
    assert de(pylcms.icc_import(ours, P("cmyk.icm")), pylcms.icc_import(theirs, P("cmyk.icm"))).max() < 3.0
    g = np.arange(256, dtype=np.uint8).reshape(-1, 1)
    assert de(host_eval(0, g, P("sGrey.icm")), pylcms.icc_import(g, P("sGrey.icm"))).max() < 0.3


def test_known_answers_and_refusals():
    """no oracle needed: white / black of an sRGB-like profile, and what the device path declines"""
    prof = F.rgb_profile()
    lab = host_eval(0, np.array([[255, 255, 255], [0, 0, 0]], np.uint8), prof)
    assert np.abs(lab - [[100, 0, 0], [0, 0, 0]]).max() < 0.02
    assert np.array_equal(host_eval(1, lab, prof), [[255, 255, 255], [0, 0, 0]])
    with pytest.raises(vb.Error, match="intent"):
        host_eval(0, np.zeros((1, 3), np.uint8), prof, intent=4)
    with pytest.raises(vb.Error, match="absolute colorimetric intent of a lut-based"):
        host_eval(0, np.zeros((1, 4), np.uint8), F.ink_profile(), intent=3)            # the scale would sit inside the evaluator
    with pytest.raises(vb.Error, match="absolute colorimetric intent of a grey"):
        host_eval(0, np.zeros((1, 1), np.uint8), F.grey_profile(), intent=3)
    with pytest.raises(vb.Error, match="lut-based"):
        host_eval(0, np.zeros((1, 4), np.uint8), F.ink_profile(), intent=0)            # needs black point compensation
    with pytest.raises(vb.Error, match="bands"):
        host_eval(0, np.zeros((1, 2), np.uint8), prof)
    with pytest.raises(vb.Error, match="ICC"):
        host_eval(0, np.zeros((1, 3), np.uint8), b"not a profile" * 20)


def test_extra_bands_ride_along():
    """vips_colour_build detaches the bands after the colour channels and re-attaches them cast to the output
    format, rescaled when the interpretations' alpha ranges differ (colour.c:196-291)"""
    prof = F.rgb_profile()
    a = np.random.default_rng(9).integers(0, 256, (500, 5), dtype=np.uint8)
    lab = host_eval(0, a, prof)
    assert lab.shape == (500, 5)
    assert np.array_equal(lab[:, :3], host_eval(0, np.ascontiguousarray(a[:, :3]), prof))
    assert np.array_equal(lab[:, 3:], a[:, 3:].astype(np.float32))              # sRGB -> Lab: both 0..255
    back = host_eval(1, lab, prof)
    assert np.array_equal(back[:, 3:], a[:, 3:]) and np.abs(back[:, :3].astype(int) - a[:, :3]).max() <= 1
    wide = host_eval(2, a, prof, F.rgb_profile("gamma"), depth=16)               # sRGB -> RGB16: alpha x 257
    assert np.array_equal(wide[:, 3:], a[:, 3:].astype(np.uint16) * 257)


@pytest.mark.gpu
def test_gpu_matches_host_evaluation(vb):
    """the kernel runs the same __host__ __device__ code: device libm pow / cbrt may move a result by an ulp,
    which can flip a rounding once in a while, never more"""
    rng = np.random.default_rng(8)
    rgb, ink, grey = F.rgb_profile(), F.ink_profile(), F.grey_profile()
    a = rng.integers(0, 256, (64, 96, 3), dtype=np.uint8)
    lab = vb.Image(a, "srgb").icc_import(rgb)
    assert lab.array.dtype == np.float32 and lab.array.shape == a.shape
    assert np.abs(lab.array.reshape(-1, 3) - host_eval(0, a.reshape(-1, 3), rgb)).max() < 2e-3
    back = lab.icc_export(rgb).numpy()
    want = host_eval(1, lab.array.reshape(-1, 3), rgb).reshape(a.shape)
    assert np.abs(back.astype(int) - want.astype(int)).max() <= 1 and (back != want).mean() < 1e-3
    assert np.abs(back.astype(int) - a.astype(int)).max() <= 1          # import then export is the identity to 1 LSB
    inks = vb.Image(a, "srgb").icc_transform(ink, rgb).numpy()
    want = host_eval(2, a.reshape(-1, 3), rgb, ink).reshape(64, 96, 4)
    assert np.abs(inks.astype(int) - want.astype(int)).max() <= 1
    c = rng.integers(0, 65536, (32, 48, 4), dtype=np.uint16)
    got = vb.Image(c, "cmyk").icc_import(ink, pcs="xyz").numpy()
    assert np.abs(got.reshape(-1, 3) - host_eval(0, c.reshape(-1, 4), ink, pcs=1)).max() < 2e-3
    rgba = rng.integers(0, 256, (24, 40, 4), dtype=np.uint8)
    got = vb.Image(rgba, "srgb").icc_transform(rgb, rgb, depth=16).numpy()
    assert got.shape == (24, 40, 4) and np.array_equal(got[..., 3], rgba[..., 3].astype(np.uint16) * 257)
    v4 = F.lut_v4_rgb_profile("Lab ")
    got = vb.Image(a, "srgb").icc_transform(v4, v4).numpy()                  # lutAtoB then lutBtoA
    want = host_eval(2, a.reshape(-1, 3), v4, v4).reshape(a.shape)
    assert np.abs(got.astype(int) - want.astype(int)).max() <= 1
    g = rng.integers(0, 256, (16, 40, 1), dtype=np.uint8)
    got = vb.Image(g, "b-w").icc_transform(rgb, grey, depth=16).numpy()
    want = host_eval(2, g.reshape(-1, 1), grey, rgb, depth=16).reshape(16, 40, 3)
    assert np.abs(got.astype(int) - want.astype(int)).max() <= 1


@pytest.mark.gpu
def test_gpu_against_lcms2_fixtures(vb):
    """the CUDA kernel against lcms2's OWN outputs (tests/golden/icc_lcms.npz, made by make_icc_golden.py through
    oracle/pylcms.py), at the tolerances the CPU tests state for the host compile of the same evaluator -- so a
    logic error the kernel and its host twin share cannot hide behind test_gpu_matches_host_evaluation"""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_icc_golden import inputs
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "icc_lcms.npz"))
    I = inputs()
    rgb, gamma, table, grey, ink = F.rgb_profile("srgb"), F.rgb_profile("gamma"), F.rgb_profile("table"), F.grey_profile(), F.ink_profile()
    v4 = F.lut_v4_rgb_profile("Lab ")

    def img(a, interp):
        return vb.Image(a.reshape(1, a.shape[0], a.shape[1]), interp)

    def flat(im):
        return im.numpy().reshape(-1, im.numpy().shape[-1])

    # import, 8-bit and float device values, Lab and XYZ PCS
    got = flat(img(I["rgb8"], "srgb").icc_import(rgb))
    assert de(got, G["import_rgb8_lab"]).max() < 0.8 and de(got, G["import_rgb8_lab"]).mean() < 0.05
    assert np.abs(flat(img(I["rgbf"], "srgb").icc_import(rgb)) - G["import_rgbf_lab"]).max() < 0.03
    assert np.abs(flat(img(I["rgb8"], "srgb").icc_import(rgb, pcs="xyz")) - G["import_rgb8_xyz"]).max() < 0.08
    assert de(flat(img(I["rgb8"], "srgb").icc_import(table)), G["import_table8_lab"]).max() < 1.6
    # export from lcms2's own Lab
    lab = img(G["import_rgb8_lab"], "lab")
    d = np.abs(flat(lab.icc_export(rgb)).astype(int) - G["export_lab_rgb8"].astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.004
    d = np.abs(flat(lab.icc_export(rgb, depth=16)).astype(int) - G["export_lab_rgb16"].astype(int))
    assert d.max() <= 128 and d.mean() < 2
    d = np.abs(flat(lab.icc_export(gamma)).astype(int) - G["export_lab_gamma8"].astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.004
    # device to device
    d = np.abs(flat(img(I["rgb8"], "srgb").icc_transform(gamma, rgb)).astype(int) - G["transform_rgb8_gamma8"].astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.03
    d = np.abs(flat(img(I["rgb16"], "rgb16").icc_transform(gamma, rgb, depth=16)).astype(int) - G["transform_rgb16_gamma16"].astype(int))
    assert d.max() <= 256 and d.mean() < 6
    # grey, CMYK (lut16), v4 lutAtoB / lutBtoA
    assert de(flat(img(I["grey8"], "b-w").icc_import(grey)), G["import_grey8_lab"]).max() < 0.3
    assert np.array_equal(flat(img(G["import_grey8_lab"], "lab").icc_export(grey)), G["export_lab_grey8"])
    assert de(flat(img(I["cmyk8"], "cmyk").icc_import(ink)), G["import_cmyk8_lab"]).max() < 1.5
    d = np.abs(flat(lab.icc_export(ink)).astype(int) - G["export_lab_cmyk8"].astype(int))
    assert d.max() <= 2 and d.mean() < 0.05
    assert de(flat(img(I["rgb8"], "srgb").icc_import(v4)), G["import_v4_rgb8_lab"]).max() < 1.6
    d = np.abs(flat(lab.icc_export(v4)).astype(int) - G["export_lab_v4_rgb8"].astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 0.005


@needs_lcms
def test_lcms2_fixtures_are_current():
    """CPU: the stored fixtures are what lcms2 gives today for the same inputs (regenerate with make_icc_golden.py)"""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_icc_golden import inputs
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "icc_lcms.npz"))
    I = inputs()
    assert np.array_equal(pylcms.icc_import(I["rgb8"], F.rgb_profile("srgb")), G["import_rgb8_lab"])
    assert np.array_equal(pylcms.icc_export(G["import_rgb8_lab"], F.ink_profile()), G["export_lab_cmyk8"])
    # and the host twin of the kernel meets the same bars against them
    assert de(host_eval(0, I["rgb8"], F.rgb_profile("srgb")), G["import_rgb8_lab"]).max() < 0.8
    d = np.abs(host_eval(1, G["import_rgb8_lab"], F.rgb_profile("srgb")).astype(int) - G["export_lab_rgb8"].astype(int))
    assert d.max() <= 1
