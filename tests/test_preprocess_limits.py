"""The pre-pass (usv_preprocess.cu: remap -> BGR2HSV -> equalizeHist(V) -> HSV2BGR -> BGR2GRAY) on every input, at its
size limits, on strided buffers and across the frame chunks of the lighting path.

  * CPU: oracle/preprocess_oracle.py pinned against cv2 on every input it claims: BGR2HSV and BGR2GRAY on all 2^24 BGR
    triples, HSV2BGR (cv2's scalar loop) on all 180 * 256 * 256 HSV triples, and remap with map1 drawn from the whole
    int16 range and map2 from the whole uint16 range (OpenCV reads its low 10 bits).
  * GPU, bit for bit against the oracle:
      - every BGR triple through the whole chain, both flavours, lighting off and under five equalisation LUTs;
      - remap taps on the edges of the kernel's in-frame fast path, maps at the int16 extremes, map2 >= 1024, and a
        1920x1080 frame with a random map;
      - row padding, inter-frame gaps, odd destination strides and misaligned destinations, through the device and the
        host entry points: the caller's source padding must not change the result, its destination padding must survive;
      - batches of 60 frames at 640x480 and 11 at 1920x1080 (two chunks of the lighting path each);
      - a frame of more than 2^24 pixels whose cumulative counts are odd and above 2^24 (no longer exact in float), and
        degenerate histograms;
      - 32767-pixel rows and columns, and what the entry points refuse.

Output buffers are filled with a sentinel first, so a pixel the kernels leave unwritten fails the comparison."""
import ctypes as C
import functools
import itertools

import numpy as np
import pytest

from oracle import preprocess_oracle as po
from unsynchronized_stereo_vision_proj325_b200 import _abi, api

FLAVOURS = (_abi.PRE_OPENCV3, _abi.PRE_OPENCV4)
SENTINEL = 0xA7


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


# ---- every input ----------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=1)
def all_bgr():
    """[4096, 4096, 3] uint8 holding each of the 2^24 BGR triples once: pixel i is (i & 255, i >> 8 & 255, i >> 16)."""
    return np.ascontiguousarray(np.arange(1 << 24, dtype="<u4").view(np.uint8).reshape(4096, 4096, 4)[..., :3])


@functools.lru_cache(maxsize=1)
def all_bgr_hsv():
    """po.bgr2hsv of all_bgr(), in row blocks (the oracle works in int64)."""
    src = all_bgr()
    return np.concatenate([po.bgr2hsv(src[y:y + 512]) for y in range(0, 4096, 512)])


@functools.lru_cache(maxsize=1)
def all_hsv():
    """[180 * 256 * 256, 3] uint8: every 8-bit HSV triple with H in [0, 180)."""
    h, s, v = np.meshgrid(np.arange(180), np.arange(256), np.arange(256), indexing="ij")
    return np.stack([h, s, v], -1).astype(np.uint8).reshape(-1, 3)


@functools.lru_cache(maxsize=2)
def gray_of_hsv(flavour):
    """[180, 256, 256] uint8: po.bgr2gray(po.hsv2bgr((h, s, v))) of every HSV triple, so that the chain's expected output
    under any LUT is a lookup."""
    hsv = all_hsv()
    step = 1 << 20
    return np.concatenate([po.bgr2gray(po.hsv2bgr(hsv[i:i + step], flavour), flavour)
                           for i in range(0, len(hsv), step)]).reshape(180, 256, 256)


def test_bgr2hsv_and_bgr2gray_on_every_triple():
    cv2 = pytest.importorskip("cv2")
    src = all_bgr()
    assert np.array_equal(all_bgr_hsv(), cv2.cvtColor(src, cv2.COLOR_BGR2HSV))
    assert np.array_equal(po.bgr2gray(src, po.OPENCV4), cv2.cvtColor(src, cv2.COLOR_BGR2GRAY))


def test_hsv2bgr_on_every_triple():
    """cv2 runs its scalar loop on a 1-pixel-wide image (its vector body is a different computation,
    oracle/preprocess_oracle.py)."""
    cv2 = pytest.importorskip("cv2")
    hsv = all_hsv()
    exp = cv2.cvtColor(np.ascontiguousarray(hsv.reshape(-1, 1, 3)), cv2.COLOR_HSV2BGR).reshape(-1, 3)
    step = 1 << 20
    for i in range(0, len(hsv), step):
        assert np.array_equal(po.hsv2bgr(hsv[i:i + step], po.OPENCV4), exp[i:i + step]), i


def test_remap_on_the_whole_map_ranges():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(351)
    h, w = 64, 96
    src = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    m1 = rng.integers(-32768, 32768, (h, w, 2)).astype(np.int16)
    near = rng.random((h, w)) < 0.5  # half the taps near the frame, where the pixels are not all zero
    m1[near] = np.stack([rng.integers(-2, w + 2, near.sum()), rng.integers(-2, h + 2, near.sum())], -1)
    m1[0, :4] = [[-32768, -32768], [32767, 32767], [-32768, 5], [w - 1, 32767]]
    m2 = rng.integers(0, 65536, (h, w)).astype(np.uint16)
    assert (m2 >= 1024).mean() > 0.9
    exp = cv2.remap(src, m1, m2, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    assert np.array_equal(po.remap_bilinear(src, m1, m2), exp)
    assert np.array_equal(po.remap_bilinear(src, m1, m2 & 1023), exp)


# ---- device runs on caller-laid-out buffers ---------------------------------------------------------------------------
def _layout_buffers(frames, layout, fill, rng):
    """Source bytes [(n-1) * sfs + h * ss] holding `frames` at the layout (ss, sfs, ds, dfs, off), padding and gaps set to
    `fill` (a byte or "random"), and destination bytes [off + (n-1) * dfs + h * ds] set to SENTINEL."""
    n, h, w = frames.shape[:3]
    ss, sfs, ds, dfs, off = layout
    total = (n - 1) * sfs + h * ss
    src = rng.integers(0, 256, total, dtype=np.uint8) if fill == "random" else np.full(total, fill, np.uint8)
    np.lib.stride_tricks.as_strided(src, shape=frames.shape, strides=(sfs, ss, 3, 1))[...] = frames
    return src, np.full(off + (n - 1) * dfs + h * ds, SENTINEL, np.uint8)


def _check_layout(dst, frames, exp, layout):
    """Every frame equals the oracle and every byte outside the frames still holds SENTINEL."""
    n, h, w = frames.shape[:3]
    ss, sfs, ds, dfs, off = layout
    got = np.lib.stride_tricks.as_strided(dst[off:], shape=(n, h, w), strides=(dfs, ds, 1))
    for k in range(n):
        assert np.array_equal(got[k], exp[k]), (layout, k)
    outside = np.ones(dst.size, bool)
    np.lib.stride_tricks.as_strided(outside[off:], shape=(n, h, w), strides=(dfs, ds, 1))[...] = False
    assert (dst[outside] == SENTINEL).all(), (layout, np.flatnonzero(outside & (dst != SENTINEL))[:8])


def _params(w, h, layout, flavour, lighting):
    ss, sfs, ds, dfs, _ = layout
    return _abi.PreprocessParams(w, h, ss, ds, sfs, dfs, int(flavour), int(bool(lighting)))


def _run_device(ctx, frames, maps, layout, flavour, lighting, fill, rng):
    torch = pytest.importorskip("torch")
    n, h, w = frames.shape[:3]
    src, dst = _layout_buffers(frames, layout, fill, rng)
    d_src, d_dst = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
    d_maps = [None if m is None else torch.from_numpy(np.ascontiguousarray(m).view(np.int16)).cuda() for m in maps]
    ctx.preprocess_device(d_src.data_ptr(), n, *[None if m is None else m.data_ptr() for m in d_maps],
                          _params(w, h, layout, flavour, lighting), d_dst.data_ptr() + layout[4],
                          torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return d_dst.cpu().numpy()


def _run_host(ctx, frames, maps, layout, flavour, lighting, fill, rng):
    n, h, w = frames.shape[:3]
    src, dst = _layout_buffers(frames, layout, fill, rng)
    maps = [None if m is None else np.ascontiguousarray(m) for m in maps]
    p = _params(w, h, layout, flavour, lighting)
    rc = api.lib().usv_preprocess_host(ctx._h, api._ptr(src), C.c_int32(n), api._ptr(maps[0]), api._ptr(maps[1]), C.byref(p),
                                       C.c_void_p(dst.ctypes.data + layout[4]))
    ctx._check(rc, "usv_preprocess_host")
    return dst


def _oracle(frames, maps, lighting, flavour):
    return [po.preprocess(f, maps[0], maps[1], lighting=lighting, flavour=flavour) for f in frames]


def _random_maps(rng, h, w, border=3):
    m1 = np.stack([rng.integers(-border, w + border, (h, w)), rng.integers(-border, h + border, (h, w))], -1).astype(np.int16)
    return m1, rng.integers(0, 65536, (h, w)).astype(np.uint16)


# ---- every BGR triple through the chain -------------------------------------------------------------------------------
# appended rows of one colour each (V = 0, 4, 20, 90, 255): five V histograms, so five equalisation LUTs
APPENDED = ((0, 0, 0), (1, 4, 3), (5, 20, 12), (40, 90, 10), (255, 255, 255))


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", FLAVOURS)
def test_every_bgr_triple_through_the_chain(ctx, flavour):
    src = all_bgr()
    blocks = range(0, 4096, 512)  # the expected frames are computed in row blocks: the oracle works in int64
    got = ctx.preprocess(src[None], lighting=False, flavour=flavour)[0]
    for y in blocks:
        assert np.array_equal(got[y:y + 512], po.bgr2gray(src[y:y + 512], flavour)), y
    rows = 1024
    batch = np.empty((len(APPENDED), 4096 + rows, 4096, 3), np.uint8)
    batch[:, :4096] = src
    for k, colour in enumerate(APPENDED):
        batch[k, 4096:] = colour
    got = ctx.preprocess(batch, lighting=True, flavour=flavour)
    assert ctx.last_kernel.startswith("rectify_hsv_hist_kernel")
    del batch
    hsv = all_bgr_hsv()
    table = gray_of_hsv(flavour)
    hist_all = np.bincount(hsv[..., 2].ravel(), minlength=256)
    luts = []
    for k, colour in enumerate(APPENDED):
        c_hsv = po.bgr2hsv(np.array([[colour]], np.uint8))[0, 0]
        hist = hist_all.copy()
        hist[c_hsv[2]] += rows * 4096
        lut = po.equalize_lut(hist)
        luts.append(lut)
        for y in blocks:
            e = hsv[y:y + 512]
            assert np.array_equal(got[k, y:y + 512], table[e[..., 0], e[..., 1], lut[e[..., 2]]]), (k, colour, y)
        assert (got[k, 4096:] == table[c_hsv[0], c_hsv[1], lut[c_hsv[2]]]).all(), (k, colour)
    # every V but the ends (0 and 255 keep their level under any of these LUTs) meets more than one V'
    luts = np.stack(luts)
    assert all(len(set(luts[:, v])) > 1 for v in range(4, 255))


# ---- remap ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flavour", FLAVOURS)
@pytest.mark.parametrize("lighting", [False, True])
def test_remap_edges_and_extreme_maps(ctx, flavour, lighting):
    """Taps on both sides of the fast path's bounds (sx, sy in {-1, 0, w-2, w-1} and their neighbours), with zero and
    nonzero fractions, maps at the int16 extremes and map2 words with bits above the 10 OpenCV reads."""
    rng = np.random.default_rng(359)
    n, h, w = 2, 23, 37
    src = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    xs = (-32768, -2, -1, 0, 1, w - 3, w - 2, w - 1, w, 32767)
    ys = (-32768, -1, 0, h - 2, h - 1, h, 32767)
    fr = ((0, 0), (0, 31), (31, 0), (31, 31), (17, 5))
    combos = list(itertools.product(xs, ys, fr))  # 350 of the 851 pixels; the rest random near the frame
    m1, m2 = _random_maps(rng, h, w, border=2)
    flat1, flat2 = m1.reshape(-1, 2), m2.reshape(-1)
    for i, (sx, sy, (fx, fy)) in enumerate(combos):
        flat1[2 * i] = (sx, sy)
        flat2[2 * i] = fy << 5 | fx | (int(rng.integers(0, 64)) << 10 if i % 2 else 0)
    got = ctx.preprocess(src, m1, m2, lighting=lighting, flavour=flavour)
    for k, e in enumerate(_oracle(src, (m1, m2), lighting, flavour)):
        assert np.array_equal(got[k], e), k


@pytest.mark.gpu
@pytest.mark.parametrize("lighting,flavour", [(True, _abi.PRE_OPENCV4), (False, _abi.PRE_OPENCV3)])
def test_full_size_random_map(ctx, lighting, flavour):
    rng = np.random.default_rng(1080)
    h, w = 1080, 1920
    src = rng.integers(0, 256, (1, h, w, 3), dtype=np.uint8)
    src[0, :, : w // 2] //= 3  # two halves of different contrast
    xs, ys = np.meshgrid(np.arange(w), np.arange(h))
    m1 = np.stack([xs + rng.integers(-4, 5, (h, w)), ys + rng.integers(-4, 5, (h, w))], -1).astype(np.int16)
    far = rng.random((h, w)) < 0.01
    m1[far] = rng.integers(-32768, 32768, (far.sum(), 2))
    m2 = rng.integers(0, 65536, (h, w)).astype(np.uint16)
    got = ctx.preprocess(src, m1, m2, lighting=lighting, flavour=flavour)[0]
    assert np.array_equal(got, po.preprocess(src[0], m1, m2, lighting=lighting, flavour=flavour))


# ---- strides and alignment ----------------------------------------------------------------------------------------------
def _layouts(w, h):
    """(src_stride, src_frame_stride, dst_stride, dst_frame_stride, d_gray byte offset)."""
    out = []
    for ss, sgap, ds, dgap, off in ((3 * w, 0, w, 0, 0),            # packed
                                    (3 * w + 1, 0, w, 0, 0),        # odd source stride
                                    (3 * w + 16, 7, w, 0, 0),       # source gaps between frames
                                    (3 * w, 0, w + 1, 0, 0),
                                    (3 * w + 5, 33, w + 3, 5, 0),   # gaps on both sides
                                    (3 * w, 0, w, 3, 1),            # destination offsets
                                    (3 * w + 2, 0, w + 3, 0, 2),
                                    (3 * w, 11, w + 1, 1, 3)):
        out.append((ss, h * ss + sgap, ds, h * ds + dgap, off))
    return out


def _stride_cases():
    """w odd: every gray row ends in a partial group and dst_stride takes every residue; w = 40: word-sized rows whose
    32-bit stores are allowed or not by the alignment of the frame base alone."""
    cases = [(37, 13, lay) for lay in _layouts(37, 13)]
    w, h = 40, 9
    for ds, dgap, off in ((40, 0, 1), (40, 0, 2), (40, 0, 3), (40, 2, 0), (44, 4, 0), (44, 0, 0)):
        cases.append((w, h, (3 * w + 4, h * (3 * w + 4) + 3, ds, h * ds + dgap, off)))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["device", "host"])
@pytest.mark.parametrize("lighting", [False, True])
def test_strides_and_alignment(ctx, entry, lighting):
    run = _run_device if entry == "device" else _run_host
    rng = np.random.default_rng(852)
    n = 3
    for i, (w, h, layout) in enumerate(_stride_cases()):
        frames = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
        frames[1] = frames[1] // 4 + 100
        maps = _random_maps(rng, h, w) if i % 2 else (None, None)
        flavour = FLAVOURS[i % 2]
        exp = _oracle(frames, maps, lighting, flavour)
        for fill in (0xFF, "random"):
            dst = run(ctx, frames, maps, layout, flavour, lighting, fill, rng)
            _check_layout(dst, frames, exp, layout)


@pytest.mark.gpu
def test_single_frame_roi_host_entry(ctx):
    """One frame whose strides describe a window of larger images (a cv::Mat ROI; the frame strides of a single frame
    are not read): the bytes around the window are the caller's."""
    rng = np.random.default_rng(7)
    h, w = 21, 33
    big = rng.integers(0, 256, (h + 4, w + 9, 3), dtype=np.uint8)
    gray = np.full((h + 4, w + 6), SENTINEL, np.uint8)
    roi = big[2:2 + h, 5:5 + w]
    for lighting in (False, True):
        gray[...] = SENTINEL
        p = _abi.PreprocessParams(w, h, big.strides[0], gray.strides[0], 0, 0, _abi.PRE_OPENCV4, int(lighting))
        rc = api.lib().usv_preprocess_host(ctx._h, C.c_void_p(roi.ctypes.data), C.c_int32(1), None, None, C.byref(p),
                                           C.c_void_p(gray[2:, 3:].ctypes.data))
        ctx._check(rc, "usv_preprocess_host")
        assert np.array_equal(gray[2:2 + h, 3:3 + w], po.preprocess(np.ascontiguousarray(roi), lighting=lighting))
        outside = np.ones(gray.shape, bool)
        outside[2:2 + h, 3:3 + w] = False
        assert (gray[outside] == SENTINEL).all()


# ---- chunks of the lighting path ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w,chunk", [(60, 480, 640, 54), (11, 1080, 1920, 8)])
def test_batches_of_two_chunks(ctx, n, h, w, chunk):
    """The HSV words of a chunk take at most 64 MiB (usv_preprocess.cu: preprocess_chunk_frames): these batches run in
    two chunks, the second partly filled. Every frame has its own histogram."""
    assert chunk == (64 << 20) // (w * h * 4) and chunk < n < 2 * chunk
    rng = np.random.default_rng(n)
    base = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    frames = np.empty((n, h, w, 3), np.uint8)
    for k in range(n):
        frames[k] = (base.astype(np.uint16) * (30 + 3 * k) >> 8) + (k * 37) % 48  # at most 206 + 47
    before = ctx.launch_count
    got = ctx.preprocess(frames, lighting=True, flavour=_abi.PRE_OPENCV4)
    assert ctx.launch_count - before == 2 * 3
    luts = set()
    for k in range(n):
        v = po.bgr2hsv(frames[k])[..., 2]
        luts.add(po.equalize_lut(np.bincount(v.ravel(), minlength=256)).tobytes())
        assert np.array_equal(got[k], po.preprocess(frames[k], lighting=True, flavour=_abi.PRE_OPENCV4)), k
    assert len(luts) == n


# ---- histogram limits ---------------------------------------------------------------------------------------------------
def _to_f32_rz(c):
    """Round-toward-zero int -> float32 (c < 2^25)."""
    c = np.asarray(c, np.int64)
    return np.where(c >= 1 << 24, c & ~1, c).astype(np.float32)


# 4200 x 4008 = 16 833 600 pixels: V = 20 (the first bin) 83 times, the cumulative counts past it are 8 000 001,
# 16 800 511 and 16 800 513, and the denominator 16 833 517: all odd and above 2^24 but the first. At 16 800 511 the
# float conversion decides the level: rounded to nearest it is 255, rounded toward zero 254.
WIDE_W, WIDE_H = 4200, 4008
WIDE_HIST = {20: 83, 100: 8000001, 170: 8800510, 200: 2, 255: WIDE_W * WIDE_H - 83 - 8000001 - 8800510 - 2}


def test_wide_histogram_needs_rounded_counts():
    """The frame of test_histogram_past_2_24 tells the two float conversions of the cumulative counts apart."""
    hist = np.zeros(256, np.int64)
    for v, c in WIDE_HIST.items():
        hist[v] = c
    lut = po.equalize_lut(hist)
    total = hist.sum()
    cs = np.cumsum(hist[21:])
    assert total > 1 << 24 and all(c % 2 and c > 1 << 24 for c in (cs[170 - 21], cs[200 - 21], total - 83))
    scale = np.float32(255) / np.float32(total - 83)
    rz = np.clip(np.rint(_to_f32_rz(cs) * scale), 0, 255).astype(np.uint8)
    assert lut[170] == 255 and rz[170 - 21] == 254


@pytest.mark.gpu
def test_histogram_past_2_24(ctx):
    rng = np.random.default_rng(2 ** 24)
    values = np.array(sorted(WIDE_HIST), np.uint8)
    colours = np.stack([values // 3, values, values.astype(int) * 2 // 3], -1).astype(np.uint8)  # V = G, saturated
    idx = np.repeat(np.arange(len(values), dtype=np.uint8), [WIDE_HIST[v] for v in values.tolist()])
    idx = rng.permutation(idx).reshape(WIDE_H, WIDE_W)
    got = ctx.preprocess(colours[idx][None], lighting=True, flavour=_abi.PRE_OPENCV4)[0]
    hsv = po.bgr2hsv(colours)
    assert np.array_equal(hsv[:, 2], values)
    hist = np.zeros(256, np.int64)
    hist[values] = [WIDE_HIST[v] for v in values.tolist()]
    hsv[:, 2] = po.equalize_lut(hist)[hsv[:, 2]]
    exp = po.bgr2gray(po.hsv2bgr(hsv, po.OPENCV4), po.OPENCV4)
    assert np.array_equal(got, exp[idx])


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", FLAVOURS)
def test_degenerate_histograms(ctx, flavour):
    """One V, two V, V = 255 and one other, and every pixel at V = 255 (the first occupied bin is the last), alone and
    in one batch."""
    rng = np.random.default_rng(255)
    h, w = 31, 45

    def frame(vs):
        v = rng.choice(np.array(vs), (h, w))
        out = np.stack([rng.integers(0, 256, (h, w)) * v // 255, v, rng.integers(0, 256, (h, w)) * v // 255], -1)
        return out.astype(np.uint8)  # V = G

    frames = np.stack([frame([77]), frame([10, 200]), frame([0, 255]), frame([254, 255]), frame([255]), frame([0])])
    for k, f in enumerate(frames):
        assert len(np.unique(f[..., 1])) == (1 if k in (0, 4, 5) else 2)
    exp = _oracle(frames, (None, None), True, flavour)
    got = ctx.preprocess(frames, lighting=True, flavour=flavour)
    for k in range(len(frames)):
        assert np.array_equal(got[k], exp[k]), k
        assert np.array_equal(ctx.preprocess(frames[k:k + 1], lighting=True, flavour=flavour)[0], exp[k]), k


# ---- size limits --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(2, 32767), (32767, 3)])
@pytest.mark.parametrize("lighting", [False, True])
def test_largest_rows_and_columns(ctx, h, w, lighting):
    rng = np.random.default_rng(h * w)
    src = rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
    src[1] //= 5
    maps = _random_maps(rng, h, w)
    for flavour in FLAVOURS:
        for m in ((None, None), maps):
            got = ctx.preprocess(src, m[0], m[1], lighting=lighting, flavour=flavour)
            for k, e in enumerate(_oracle(src, m, lighting, flavour)):
                assert np.array_equal(got[k], e), (flavour, m[0] is not None, k)


@pytest.mark.gpu
def test_refused_arguments(ctx):
    for shape in ((1, 2, 32768, 3), (1, 32768, 2, 3)):
        with pytest.raises(api.UsvError, match="bad frame size"):
            ctx.preprocess(np.zeros(shape, np.uint8), lighting=True)
    src = np.zeros((1, 4, 5, 3), np.uint8)
    m1, m2 = np.zeros((4, 5, 2), np.int16), np.zeros((4, 5), np.uint16)
    for a, b in ((m1, None), (None, m2)):
        p = _abi.PreprocessParams(5, 4, 15, 5, 60, 20, _abi.PRE_OPENCV4, 1)
        rc = api.lib().usv_preprocess_host(ctx._h, api._ptr(src), C.c_int32(1), api._ptr(a), api._ptr(b), C.byref(p),
                                           api._ptr(np.zeros(20, np.uint8)))
        assert rc == _abi.USV_ERR_INVALID_ARG and b"come as a pair" in api.lib().usv_last_error(ctx._h)
        rc = api.lib().usv_preprocess_device(ctx._h, None, C.c_int32(1), api._ptr(a), api._ptr(b), C.byref(p), None, None)
        assert rc == _abi.USV_ERR_INVALID_ARG and b"come as a pair" in api.lib().usv_last_error(ctx._h)
    # no frames: nothing is read, written or launched
    gray = np.full(20, SENTINEL, np.uint8)
    before = ctx.launch_count
    p = _abi.PreprocessParams(5, 4, 15, 5, 60, 20, _abi.PRE_OPENCV4, 1)
    assert api.lib().usv_preprocess_host(ctx._h, None, C.c_int32(0), None, None, C.byref(p), api._ptr(gray)) == 0
    assert api.lib().usv_preprocess_device(ctx._h, None, C.c_int32(0), None, None, C.byref(p), None, None) == 0
    assert ctx.launch_count == before and (gray == SENTINEL).all()
    p.width = 32768
    assert api.lib().usv_preprocess_device(ctx._h, None, C.c_int32(0), None, None, C.byref(p), None, None) == _abi.USV_ERR_INVALID_ARG
