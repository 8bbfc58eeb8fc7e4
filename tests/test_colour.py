"""Colour path.  CPU: the oracle against the reference's own line functions
(oracle/_ref, or its outputs' stored digests: tests/refgold.py) and the known answers in the reference's test_colour.py.  GPU:
the fused route kernel against the oracle, bit for bit (the spec allows 1 ULP
on float; we assert 0) through the C ABI.
"""
import numpy as np
import pytest

from oracle import pyoracle as orc
from oracle import pyref
from refgold import ref  # noqa: F401

SPACES = ["srgb", "scrgb", "xyz", "lab", "labs", "rgb16"]
SPACE_DT = {"srgb": np.uint8, "rgb16": np.uint16, "labs": np.int16, "scrgb": np.float32, "xyz": np.float32,
            "lab": np.float32}


def sample(space, rng, n=20000, wild=False):
    if space == "srgb":
        return rng.integers(0, 256, (n, 3), dtype=np.uint8)
    if space == "rgb16":
        return rng.integers(0, 65536, (n, 3), dtype=np.uint16)
    if space == "labs":
        a = rng.integers(-32768, 32768, (n, 3), dtype=np.int64).astype(np.int16)
        a[:, 0] = np.abs(a[:, 0])
        return a
    if wild:
        a = (rng.standard_normal((n, 3)) * 150).astype(np.float32)
        a[::97, 0] = np.nan
        a[::89, 1] = np.inf
        a[::83, 2] = -np.inf
        return a
    if space == "scrgb":
        return rng.random((n, 3), dtype=np.float32) * 1.2 - 0.1
    if space == "xyz":
        return rng.random((n, 3), dtype=np.float32) * 110 - 5
    lab = rng.random((n, 3), dtype=np.float32)
    lab[:, 0] *= 100
    lab[:, 1:] = lab[:, 1:] * 256 - 128
    return lab


STEP_SPACE = [("sRGB2scRGB", "srgb"), ("RGB162scRGB", "rgb16"), ("scRGB2XYZ", "scrgb"), ("XYZ2Lab", "xyz"),
              ("Lab2LabS", "lab"), ("LabS2Lab", "labs"), ("Lab2XYZ", "lab"), ("XYZ2scRGB", "xyz"),
              ("scRGB2sRGB", "scrgb"), ("scRGB2RGB16", "scrgb")]


def test_tables_match_reference(ref):
    for which in range(5):
        ref.check(orc.colour_table(which), lambda: pyref.colour_table(which))


@pytest.mark.parametrize("step,space", STEP_SPACE)
def test_oracle_step_matches_reference_line(ref, step, space):
    rng = np.random.default_rng(7)
    for wild in (False, True):
        a = sample(space, rng, wild=wild)
        got = orc.colour_step(a.reshape(1, -1, 3), step, space).reshape(-1, 3)
        ref.check(got, lambda: pyref.colour_line(step, a), step)


def test_known_answer_lab_to_xyz():
    """test_colour.py:53-57: Lab(50,0,0) -> XYZ = [17.5064, 18.4187, 20.0547] (Lindbloom)"""
    xyz = orc.colourspace(np.array([[[50, 0, 0]]], np.float32), "xyz", "lab").ravel()
    assert np.allclose(xyz, [17.5064, 18.4187, 20.0547], atol=1e-4)


def test_oracle_all_pairs_round_trip():
    """test_colour.py:9-51: every pair of spaces round-trips Lab(50,0,0) + alpha 42 within 0.1"""
    start = np.array([[[50, 0, 0, 42]]], np.float32)
    for a in SPACES:
        x = orc.colourspace(start, a, "lab")
        for b in SPACES:
            y = orc.colourspace(x, b, a)
            back = orc.colourspace(y, "lab", b).astype(np.float64).ravel()
            tol = 0.5 if "srgb" in (a, b) else 0.1  # 8-bit quantisation
            assert np.abs(back[:3] - [50, 0, 0]).max() < tol, (a, b, back)
            assert abs(back[3] - 42) < 1.0, (a, b, back)


def test_srgb_all_triples_round_trip_exact():
    """sRGB -> Lab -> sRGB is the identity on 8-bit data (BASELINE config 4 property)"""
    rng = np.random.default_rng(1)
    a = rng.integers(0, 256, (64, 4096, 3), dtype=np.uint8)
    lab = orc.colourspace(a, "lab", "srgb")
    assert lab.dtype == np.float32
    assert np.array_equal(orc.colourspace(lab, "srgb", "lab"), a)


# ---------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("src", SPACES)
@pytest.mark.parametrize("dst", SPACES)
def test_gpu_routes(vb, src, dst):
    rng = np.random.default_rng(11)
    a = sample(src, rng, n=64 * 257).reshape(64, 257, 3)
    got = vb.Image(a, src).colourspace(dst).numpy()
    want = orc.colourspace(a, dst, src)
    assert got.dtype == want.dtype == SPACE_DT[dst]
    assert np.array_equal(got, want, equal_nan=True), (src, dst, np.nanmax(np.abs(got.astype(np.float64) - want)))


@pytest.mark.gpu
@pytest.mark.parametrize("src", ["scrgb", "xyz", "lab"])
def test_gpu_wild_floats(vb, src):
    """NaN / Inf / out-of-gamut inputs follow the reference's clipping"""
    rng = np.random.default_rng(12)
    a = sample(src, rng, n=40000, wild=True).reshape(100, 400, 3)
    for dst in SPACES:
        got = vb.Image(a, src).colourspace(dst).numpy()
        want = orc.colourspace(a, dst, src)
        assert np.array_equal(got, want, equal_nan=True), (src, dst)


@pytest.mark.gpu
@pytest.mark.parametrize("bands", [4, 5])
def test_gpu_extra_bands(vb, bands):
    """alpha rides along: rescaled by max_alpha ratio and cast per step (colour.c:252-291)"""
    rng = np.random.default_rng(13)
    for src in SPACES:
        rgb = sample(src, rng, n=33 * 65)
        extra = sample(src, rng, n=33 * 65)[:, :bands - 3]
        a = np.concatenate([rgb, extra], axis=1).reshape(33, 65, bands)
        for dst in SPACES:
            got = vb.Image(a, src).colourspace(dst).numpy()
            want = orc.colourspace(a, dst, src)
            assert np.array_equal(got, want, equal_nan=True), (src, dst)


@pytest.mark.gpu
def test_gpu_srgb_lab_round_trip_full_gamut(vb):
    """BASELINE config 4 at reduced size: all 2^24 sRGB triples -> Lab -> sRGB is exact,
    and Lab equals the oracle's on a sample"""
    g = np.arange(256, dtype=np.uint8)
    a = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(4096, 4096, 3)
    lab = vb.Image(a, "srgb").colourspace("lab")
    back = lab.colourspace("srgb").numpy()
    assert np.array_equal(back, a)
    assert np.array_equal(lab.numpy()[:64], orc.colourspace(a[:64], "lab", "srgb"))


# ------------------------------------------------------------------ SURVEY 8f rank 3: Lab <-> LCh, XYZ <-> Yxy
NEW_STEPS = [("Lab2LCh", "lab"), ("LCh2Lab", "lch"), ("XYZ2Yxy", "xyz"), ("Yxy2XYZ", "yxy")]


def sample_new(space, rng, n=20000):
    if space == "lch":
        a = rng.random((n, 3), dtype=np.float32)
        a[:, 0] *= 100
        a[:, 1] *= 130
        a[:, 2] *= 360
        return a
    if space == "yxy":
        a = rng.random((n, 3), dtype=np.float32)
        a[:, 0] *= 100
        a[::50, 1] = 0
        a[::70, 2] = 0
        return a
    a = sample(space, rng, n)
    if space == "lab":
        a[::40, 1] = 0          # the hue's quadrant cases (Lab2LCh.c:68-75)
        a[::80, 2] = 0
    if space == "xyz":
        a[::60] = 0             # total == 0 (XYZ2Yxy.c:74-77)
    return a


@pytest.mark.parametrize("step,space", NEW_STEPS)
def test_oracle_new_converters_match_reference_lines(ref, step, space):
    """the reference's own Lab2LCh.c / LCh2Lab.c / XYZ2Yxy.c / Yxy2XYZ.c under oracle/_ref (same glibc: bit for bit)"""
    a = sample_new(space, np.random.default_rng(17))
    got = orc.colour_step(a.reshape(1, -1, 3), step, space).reshape(-1, 3)
    ref.check(got, lambda: pyref.colour_line(step, a))


def test_new_spaces_routes_follow_the_table():
    """colourspace.c:226, 236, 242, 252, 275-290: LCH hangs off LAB, YXY off XYZ"""
    L = orc.lib()
    import ctypes as C
    steps = (C.c_int * 8)()
    name = {v: k for k, v in orc.STEPS.items()}
    rows = {("srgb", "lch"): ["sRGB2scRGB", "scRGB2XYZ", "XYZ2Lab", "Lab2LCh"], ("lch", "srgb"): ["LCh2Lab", "Lab2XYZ", "XYZ2scRGB", "scRGB2sRGB"],
            ("lab", "yxy"): ["Lab2XYZ", "XYZ2Yxy"], ("yxy", "lch"): ["Yxy2XYZ", "XYZ2Lab", "Lab2LCh"], ("labs", "lch"): ["LabS2Lab", "Lab2LCh"],
            ("lch", "labs"): ["LCh2Lab", "Lab2LabS"], ("xyz", "lch"): ["XYZ2Lab", "Lab2LCh"], ("lch", "yxy"): ["LCh2Lab", "Lab2XYZ", "XYZ2Yxy"]}
    for (a, b), want in rows.items():
        n = L.orc_colourspace_route(orc.SPACES[a], orc.SPACES[b], steps)
        assert [name[steps[i]] for i in range(n)] == want, (a, b)


ALL_SPACES = SPACES + ["lch", "yxy"]


@pytest.mark.parametrize("bands", [3, 4, 5])
def test_oracle_colourspace_matches_reference_build(ref, bands):
    """the whole of vips_colourspace, not only the line functions: colourspace.c's route table and build, a real VipsColour
    object per step (colour.c: extra bands detached, alpha rescaled by the max_alpha ratio through linear.c, cast through
    cast.c and re-attached; the input casts of VipsColourCode / VipsColourTransform), vips_colour_gen pulling tiles --
    all compiled in place under oracle/ref_shim -- against the oracle's restatement, every pair of the 8 spaces"""
    rng = np.random.default_rng(30 + bands)
    for src in ALL_SPACES:
        base = "lab" if src in ("lch", "yxy") else src
        a = sample(base, rng, n=31 * 47)
        if bands > 3:
            a = np.concatenate([a, sample(base, rng, n=31 * 47)[:, :bands - 3]], axis=1)
        a = a.reshape(31, 47, bands)
        for dst in ALL_SPACES:
            got = orc.colourspace(a, dst, src)
            ref.check(got, lambda: pyref.RefImage.from_array(a, orc.SPACES[src]).colourspace(dst, src).numpy(tile=(16, 8)),
                      (src, dst, bands))


def test_oracle_colourspace_wild_floats_and_foreign_formats_match_reference_build(ref):
    """NaN / Inf pixels AND alpha through the reference's builds (alpha: linear.c then cast.c's float -> int clip), and
    images whose band format is not the one their interpretation implies (the reference casts the whole image first:
    colour.c:338-347, 421-428)"""
    rng = np.random.default_rng(41)
    for bands in (3, 4):
        for src in ("scrgb", "xyz", "lab", "lch", "yxy"):
            a = sample("lab", rng, n=23 * 40, wild=True)
            if bands > 3:
                a = np.concatenate([a, sample("lab", rng, n=23 * 40, wild=True)[:, :1]], axis=1)
            a = a.reshape(23, 40, bands)
            for dst in ALL_SPACES:
                ref.check(orc.colourspace(a, dst, src), lambda: pyref.RefImage.from_array(a, orc.SPACES[src]).colourspace(dst, src).numpy(),
                          (src, dst, bands))
    declined = 0
    for dt in (np.uint8, np.uint16, np.int16, np.int32, np.float32):
        if dt == np.float32:
            a = (rng.standard_normal((19, 21, 4)) * 200).astype(np.float32)
        else:
            a = rng.integers(np.iinfo(dt).min, np.iinfo(dt).max + 1, (19, 21, 4)).astype(dt)
        for src in ALL_SPACES:
            for dst in ALL_SPACES:
                try:
                    got = orc.colourspace(a, dst, src)
                except ValueError:
                    # the one thing not restated: a shifting cast from a format that is neither uchar nor ushort
                    assert {src, dst} == {"srgb", "rgb16"} and dt not in (np.uint8, np.uint16), (dt, src, dst)
                    declined += 1
                    continue
                ref.check(got, lambda: pyref.RefImage.from_array(a, orc.SPACES[src]).colourspace(dst, src).numpy(), (dt, src, dst))
    assert declined == 6


def test_srgb_rgb16_rows_are_shifting_casts(ref):
    """colourspace.c:372, 420: sRGB <-> RGB16 never touch the scRGB tables -- vips_cast(shift) over every band, alpha too:
    up, the bottom bit fills the new byte (cast.c:150-164); down, the high byte"""
    v = np.arange(256, dtype=np.uint8)
    a = np.stack([v, v[::-1], v, v], axis=1).reshape(16, 16, 4)
    up = orc.colourspace(a, "rgb16", "srgb")
    assert np.array_equal(up, (a.astype(np.uint16) << 8) | np.where(a & 1, 255, 0).astype(np.uint16))
    ref.check(up, lambda: pyref.RefImage.from_array(a, 22).colourspace("rgb16", "srgb").numpy())
    ref.check(up, lambda: pyref.RefImage.from_array(a, 22).cast(np.uint16, shift=True).numpy())
    w = np.arange(65536, dtype=np.uint16).reshape(256, 64, 4)
    down = orc.colourspace(w, "srgb", "rgb16")
    assert np.array_equal(down, (w >> 8).astype(np.uint8))
    ref.check(down, lambda: pyref.RefImage.from_array(w, 25).colourspace("srgb", "rgb16").numpy())
    L, steps = orc.lib(), (__import__("ctypes").c_int * 8)()
    assert L.orc_colourspace_route(22, 25, steps) == 1 and steps[0] == orc.STEPS["sRGB2RGB16"]
    assert L.orc_colourspace_route(25, 22, steps) == 1 and steps[0] == orc.STEPS["RGB162sRGB"]


def ulp_diff(a, b):
    """distance in float32 ULPs (both finite, same sign or zero)"""
    ia = a.view(np.int32).astype(np.int64)
    ib = b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7fffffff), ia)
    ib = np.where(ib < 0, -(ib & 0x7fffffff), ib)
    return np.abs(ia - ib)


@pytest.mark.gpu
@pytest.mark.parametrize("src,dst", [("xyz", "yxy"), ("yxy", "xyz"), ("srgb", "yxy"), ("yxy", "srgb"), ("yxy", "lab"), ("rgb16", "yxy")])
def test_gpu_yxy_routes_exact(vb, src, dst):
    rng = np.random.default_rng(21)
    a = (sample_new(src, rng, 64 * 129) if src in ("yxy", "xyz") else sample(src, rng, 64 * 129)).reshape(64, 129, 3)
    got = vb.Image(a, src).colourspace(dst).numpy()
    want = orc.colourspace(a, dst, src)
    assert got.dtype == want.dtype and np.array_equal(got, want, equal_nan=True), (src, dst)


@pytest.mark.gpu
@pytest.mark.parametrize("src,dst", [("lab", "lch"), ("lch", "lab"), ("srgb", "lch"), ("lch", "srgb"), ("lch", "yxy"), ("labs", "lch")])
def test_gpu_lch_routes_within_one_ulp(vb, src, dst):
    """atan / cosf / sinf: CUDA's libm against the reference's glibc -- float results within 1 ULP (cos / sin: 2), the
    tolerance north_star sets for the float colour path; integer outputs within 1 code"""
    rng = np.random.default_rng(22)
    a = (sample_new(src, rng, 64 * 129) if src in ("lch", "lab") else sample(src, rng, 64 * 129)).reshape(64, 129, 3)
    got = vb.Image(a, src).colourspace(dst).numpy()
    want = orc.colourspace(a, dst, src)
    assert got.dtype == want.dtype and got.shape == want.shape
    if want.dtype == np.float32:
        # an angle near 0 / 360 or a cosine near 0 makes "ULP" meaningless: compare with an absolute floor
        d = np.abs(got.astype(np.float64) - want)
        ok = (ulp_diff(got, want) <= (2 if src == "lch" else 1)) | (d < 2e-5)
        if (src, dst) == ("lch", "yxy"):
            # two more steps after the trigonometric one.  Lab2XYZ cubes its input: the last-place difference of
            # cosf / sinf grows to a few ULP of XYZ -- still 1e-5 relative.  XYZ2Yxy then divides by X + Y + Z, which the
            # wild samples bring arbitrarily close to zero, so a bound on x / y themselves would be a bound on luck:
            # hold XYZ to the tolerance, and Yxy to the (exact, test_gpu_yxy_routes_exact) last step applied to the
            # device's own XYZ -- the fused route keeps float intermediates exactly like the reference's float images
            got_xyz = vb.Image(a, src).colourspace("xyz").numpy()
            want_xyz = orc.colourspace(a, "xyz", src)
            dx = np.abs(got_xyz.astype(np.float64) - want_xyz)
            okx = (ulp_diff(got_xyz, want_xyz) <= 8) | (dx <= 1e-5 * np.maximum(np.abs(want_xyz), 1.0))
            assert okx.all(), (src, "xyz", dx.max())
            assert np.array_equal(got, orc.colourspace(got_xyz, "yxy", "xyz"), equal_nan=True)
            assert (got == want).mean() > 0.8
            return
        assert ok.all(), (src, dst, d.max())
        # cosf / sinf differ from glibc's in the last place on ~1 value in 9; the double atan() path on < 1 in 100
        assert (got == want).mean() > (0.8 if src == "lch" else 0.99)
    else:
        assert np.abs(got.astype(int) - want.astype(int)).max() <= 1
