"""GPU parity of the pre-pass (usv_preprocess.cu; reference P/Main.cpp:914-921) against the numpy oracle, which is
itself pinned against cv2 (tests/test_preprocess_oracle.py), and against the cv2 golden vectors directly. Bit-exact."""
import os

import numpy as np
import pytest

from oracle import preprocess_oracle as po
from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "preprocess_cv2.npz"))


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def test_golden_chain_equals_cv2(ctx):
    got = ctx.preprocess(G["src"][None], G["map1"], G["map2"], lighting=True, flavour=_abi.PRE_OPENCV4)[0]
    assert np.array_equal(got, G["gray"])
    assert ctx.last_kernel.startswith("rectify_hsv_hist_kernel")
    plain = ctx.preprocess(G["src"][None], G["map1"], G["map2"], lighting=False, flavour=_abi.PRE_OPENCV4)[0]
    assert np.array_equal(plain, G["gray_plain"])
    assert ctx.last_kernel == "rectify_gray_kernel"


@pytest.mark.parametrize("flavour", [_abi.PRE_OPENCV3, _abi.PRE_OPENCV4])
@pytest.mark.parametrize("lighting", [False, True])
def test_batches_random_maps_and_odd_sizes(ctx, flavour, lighting):
    rng = np.random.default_rng(914)
    for (n, h, w) in ((3, 33, 47), (2, 64, 128), (5, 17, 5), (1, 1, 1)):
        src = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
        src[0] = (src[0] // 4 + 60)                      # a low-contrast frame: the equalisation has work to do
        if n > 1:
            src[1] = 77                                  # a flat frame: degenerate histogram (OpenCV: setTo)
        m1 = np.stack([rng.integers(-3, w + 3, (h, w)), rng.integers(-3, h + 3, (h, w))], -1).astype(np.int16)
        m2 = rng.integers(0, 1024, (h, w)).astype(np.uint16)
        for maps in ((None, None), (m1, m2)):
            got = ctx.preprocess(src, maps[0], maps[1], lighting=lighting, flavour=flavour)
            for k in range(n):
                exp = po.preprocess(src[k], maps[0], maps[1], lighting=lighting, flavour=flavour)
                assert np.array_equal(got[k], exp), (n, h, w, k, maps[0] is not None)


def test_hsv2bgr_all_hues(ctx):
    """Random frames whose pixels take every hue H in [0, 180) at many saturations and values go through the device
    HSV2BGR, under the equalisation LUT of each frame. (Every BGR triple, and so every (H, S, V) that BGR2HSV can give,
    goes through the chain in test_preprocess_limits.py.)"""
    rng = np.random.default_rng(5)
    src = rng.integers(0, 256, (4, 256, 256, 3), dtype=np.uint8)
    for k in range(4):
        assert len(np.unique(po.bgr2hsv(src[k])[..., 0])) == 180
    for fl in (_abi.PRE_OPENCV3, _abi.PRE_OPENCV4):
        got = ctx.preprocess(src, lighting=True, flavour=fl)
        for k in range(4):
            assert np.array_equal(got[k], po.preprocess(src[k], lighting=True, flavour=fl))


def test_identity_map_and_full_size(ctx):
    """1920x1080 batch: an identity rectification map changes nothing; two runs give identical bytes; rows padded to 16."""
    n, h, w = 3, 1080, 1920
    rng = np.random.default_rng(2)
    src = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    xs, ys = np.meshgrid(np.arange(w, dtype=np.int16), np.arange(h, dtype=np.int16))
    m1, m2 = np.stack([xs, ys], -1), np.zeros((h, w), np.uint16)
    a = ctx.preprocess(src, None, None, lighting=True)
    b = ctx.preprocess(src, m1, m2, lighting=True)
    assert np.array_equal(a, b) and np.array_equal(a, ctx.preprocess(src, m1, m2, lighting=True))
    assert np.array_equal(a[1, 500:520], po.preprocess(src[1], lighting=True)[500:520])


def test_prepass_feeds_the_block_search(ctx, oracle):
    """Camera frames -> pre-pass -> dense block search, all on the device path; the known shift is recovered."""
    left_g, right_g = synth.make_pairs(1, 320, 64, 3, shift=21, noise_sigma=0.0, seed=3)
    gl = ctx.preprocess(np.ascontiguousarray(left_g), lighting=False)
    gr = ctx.preprocess(np.ascontiguousarray(right_g), lighting=False)
    assert np.array_equal(gl[0], po.bgr2gray(left_g[0]))
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_max=63)
    got = ctx.match_dense(gl, gr, p, mask=_abi.OUT_DISPARITY_U16 | _abi.OUT_RAW_COST)
    exp = oracle.match_dense(gl, gr, p, mask=_abi.OUT_DISPARITY_U16 | _abi.OUT_RAW_COST)
    assert np.array_equal(got["disparity_u16"], exp["disparity_u16"]) and np.array_equal(got["raw_cost"], exp["raw_cost"])
    nx = 320 - 15
    assert (got["disparity_u16"][0].reshape(-1, nx)[:, 21:] == 21).mean() > 0.99
