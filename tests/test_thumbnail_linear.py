"""linear=TRUE thumbnails (SURVEY 3.1b): sRGB -> scRGB, float premultiply / resize /
unpremultiply, scRGB -> sRGB.  Known answer from the reference's test-suite
(test_resample.py:234-238) + GPU parity against the oracle."""
import os

import numpy as np
import pytest

from refgold import ref  # noqa: F401

HERE = os.path.dirname(os.path.abspath(__file__))
FIX = np.load(os.path.join(HERE, "golden", "rgba_fixture.npz"))


def flatten_avg(t):
    t = t.astype(np.float64)
    al = t[..., 3:4] / 255.0
    return float((t[..., :3] * al + 255.0 * (1 - al)).mean())


def test_oracle_rgba_correct_known_answer(oracle):
    t = oracle.thumbnail_image(FIX["rgba"], 64, linear=True)
    assert t.shape[:2] == tuple(FIX["correct_shape"][:2])
    assert abs(flatten_avg(t) - float(FIX["correct_avg"])) < 1


@pytest.mark.gpu
def test_gpu_rgba_correct_known_answer(vb, oracle):
    t = vb.Image(FIX["rgba"]).thumbnail_image(64, linear=True).numpy()
    assert abs(flatten_avg(t) - float(FIX["correct_avg"])) < 1
    assert np.array_equal(t, oracle.thumbnail_image(FIX["rgba"], 64, linear=True))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,target,bands", [((512, 512), 64, 4), ((301, 517), 50, 4), ((400, 300), 60, 3),
                                                 ((640, 480), 111, 4)])
def test_gpu_linear_thumbnail_parity(vb, oracle, shape, target, bands):
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, shape + (bands,), dtype=np.uint8)
    got = vb.Image(a).thumbnail_image(target, linear=True).numpy()
    want = oracle.thumbnail_image(a, target, linear=True)
    assert got.shape == want.shape and np.array_equal(got, want)


def test_oracle_linear_chain_against_reference_sources(ref):
    """CPU: the oracle's linear-light thumbnail against the reference's OWN sources under oracle/_ref --
    premultiply.c, resize.c (shrinkv / reducev / shrinkh / reduceh float branches), unpremultiply.c and the
    sRGB2scRGB / scRGB2sRGB line functions; only the 4th band's trip through vips_colour_build (x 1 / 255,
    x 255, cast) is restated here (colour.c:252-291)."""
    from oracle import pyref
    from oracle import pyoracle as orc

    def reference(a, target):
        h, w, b = a.shape
        hs, vs, _, _ = orc.thumbnail_size(w, h, target)
        lin = pyref.colour_line("sRGB2scRGB", a[:, :, :3]).reshape(h, w, 3)
        if b == 4:
            alpha = (np.float32(1.0 / 255.0) * a[:, :, 3].astype(np.float32) + np.float32(0)).astype(np.float32)
            lin = np.concatenate([lin, alpha[:, :, None]], axis=2)
        im = pyref.RefImage.from_array(np.ascontiguousarray(lin), 28)
        if b == 4:
            im = im.premultiply()
        im = im.resize(1.0 / hs, 1.0 / vs)
        if b == 4:
            im = im.unpremultiply()
        res = im.numpy()
        rgb = pyref.colour_line("scRGB2sRGB", np.ascontiguousarray(res[:, :, :3])).reshape(res.shape[0], res.shape[1], 3)
        if b == 4:
            al = np.clip((np.float32(255.0) * res[:, :, 3] + np.float32(0)).astype(np.float32).astype(np.float64), 0, 255).astype(np.uint8)
            rgb = np.concatenate([rgb, al[:, :, None]], axis=2)
        return rgb
    rng = np.random.default_rng(77)
    for shape, target in (((256, 320, 4), 40), ((200, 150, 3), 33), ((333, 222, 4), 60)):
        a = rng.integers(0, 256, shape, dtype=np.uint8)
        ref.check(orc.thumbnail_image(a, target, linear=True), lambda: reference(a, target), shape)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,target,bands", [((2048, 2048), 256, 4), ((1024, 768), 128, 4), ((1200, 900), 150, 4),
                                                 ((1003, 2057), 120, 4), ((777, 555), 99, 3), ((4096, 512), 64, 4)])
def test_gpu_linear_two_kernel_path(vb, oracle, shape, target, bands):
    """the geometries of the uchar V4 cases through the linear-light kernels, and that they ARE the kernels"""
    rng = np.random.default_rng(6)
    a = rng.integers(0, 256, shape + (bands,), dtype=np.uint8)
    a[: shape[0] // 3, :, -1] = 0  # transparent band: unpremultiply's |alpha| < 0.01 branch
    plan = vb.ThumbnailPlan(shape[1], shape[0], bands, target, linear=True)
    assert plan.fused and plan.kernel == "linear_v_kernel + linear_h_kernel"
    n0 = vb.launch_count()
    got = plan.run_host(a[None])[0]
    assert vb.launch_count() - n0 == 2
    want = oracle.thumbnail_image(a, target, linear=True)
    assert got.shape == want.shape and np.array_equal(got, want)


@pytest.mark.gpu
def test_gpu_linear_batch_and_sharpen_stage(vb, oracle):
    from oracle import pyconv
    rng = np.random.default_rng(8)
    frames = rng.integers(0, 256, (5, 600, 800, 4), dtype=np.uint8)
    plan = vb.ThumbnailPlan(800, 600, 4, 100, linear=True)
    got = plan.run_host(frames)
    for i in range(5):
        assert np.array_equal(got[i], oracle.thumbnail_image(frames[i], 100, linear=True)), i
    plan.set_sharpen()
    got = plan.run_host(frames[:2])
    for i in range(2):
        assert np.array_equal(got[i], pyconv.sharpen(oracle.thumbnail_image(frames[i], 100, linear=True), "srgb")), i
