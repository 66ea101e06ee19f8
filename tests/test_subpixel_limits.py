"""The sub-pixel pass (usv_subpixel.cu, DESIGN §4.8) at every cost and channel count, at its integer limits and on
refinement targets the caller chooses.

The refinement is specified for any RightIndex a caller hands it (include/usv_b200.h), not only for the sweep's own
winners, and only caller-chosen targets reach every arm of it: the +-8 clamp, den = 0 and den < 0 in the int64 and in
the f64 arm, a neighbour outside the clipped range (q = 0) and targets that are no candidate (NO_SUBPIXEL).

  * CPU: tests/subpixel_oracle.c against the restatement of test_subpixel.py on such targets, with the count of every
    arm checked independently from int64 / f64 costs computed here (`classify`). This pins the oracle first.
  * GPU: usv_refine_subpixel_device called directly on device frames and a device RightIndex built by the test, bit for
    bit against the oracle: the same targets at C = 1..4; 32768-byte templates for SAD / SSD / NCC / ZNCC at every C,
    where an SSD cost reaches 65025 * 32768 and c(x*-1) + c(x*+1) passes 2^31 (it cannot pass 2^32: two costs are at
    most 4 261 478 400); template rows of one word and of 1024 bytes, every residue of tw*C mod 4, th = 1, strides
    1..3, grids wider than one 128-window CTA, three pairs with a gap between frames, dirty row padding, and a grid of
    more than 65535 window rows (the kernel's grid-stride row loop); each output pointer alone; DIST_NONE.
  * GPU: all 16 <cost, C> instances behind the sweep that serves them (usv_last_kernel checked), the host entry point at
    C = 2 and 4 with an odd host row stride, and ~100 seeded random configurations whose targets mix the sweep's winners
    with perturbed ones.

Outputs are pre-filled with a sentinel, so a window the kernel leaves unwritten fails the comparison. The comparison
rule is test_subpixel.py's: disparity_x16 equal, PINHOLE distances byte-equal, POWERLAW distances to rtol 1e-12 with
the same zero and NaN positions (the device's pow may differ from the host's in the last bit)."""
import math
import os
import subprocess

import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth
from test_gpu_limits import _scores, pattern
from test_subpixel import SubpixelOracle, restate

COSTS = ("sad", "ssd", "ncc", "zncc")
SIDES = (_abi.LEFT_CAM, _abi.RIGHT_CAM)
UNBOUNDED = 1 << 20
X16_SENTINEL = 0x5A5A5A5A  # never a refined disparity of these frames
DIST_SENTINEL = 12345.678  # never a distance of these frames

# arms of the refinement (classify)
NONE, EDGE, DEN0, DENNEG, CLAMP_P, CLAMP_M, FIT = range(7)
ARM_NAMES = ("not a candidate", "neighbour outside the range", "den = 0", "den < 0", "clamped to +8", "clamped to -8",
             "inside +-8")


@pytest.fixture(scope="module")
def sub(tmp_path_factory):
    here = os.path.dirname(os.path.abspath(__file__))
    so = str(tmp_path_factory.mktemp("subpixel_oracle") / "libusv_subpixel_oracle.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"  # as oracle/Makefile: the system compiler has OpenMP
    out = subprocess.run([cc, "-O3", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-o", so,
                          os.path.join(here, "subpixel_oracle.c"), "-lm"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return SubpixelOracle(so)


# ---- geometry, targets and the arm of every window ------------------------------------------------------------------
def _geometry(shape, p):
    """(nx, ny, nxc, nyc, x [nwin], y [nwin], lo [nwin], hi [nwin]) of frames [n, H, W(, C)]; lo > hi: empty range."""
    h, w = shape[1], shape[2]
    nxc, nyc = w - p.tmpl_w + 1, h - p.tmpl_h + 1
    nx, ny = (nxc - 1) // p.stride_x + 1, (nyc - 1) // p.stride_y + 1
    k = np.arange(nx * ny, dtype=np.int64)
    x, y = (k % nx) * p.stride_x, (k // nx) * p.stride_y
    if p.camera_side == _abi.LEFT_CAM:
        lo, hi = x - p.search_max, x - p.search_min
    else:
        lo, hi = x + p.search_min, x + p.search_max
    return nx, ny, nxc, nyc, x, y, np.maximum(lo, 0), np.minimum(hi, nxc - 1)


def targets(shape, p, rng, n=None, foreign=0.15):
    """RightIndex [n, ny*nx] a caller might pass: x* spread over the window's range and two pixels past either end,
    x* = 1 and x* = nxc - 2 (the candidates whose neighbour is the first / last position of the row), and a `foreign`
    share of non-candidates: NO_MATCH, a candidate of the next window row, an index past the frame, 0xFFFFFFFE."""
    n = shape[0] if n is None else n
    nx, ny, nxc, nyc, x, y, lo, hi = _geometry(shape, p)
    nwin = nx * ny
    out = np.empty((n, nwin), np.int64)
    for i in range(n):
        span = np.maximum(hi - lo + 5, 1)
        xs = lo - 2 + (rng.random(nwin) * span).astype(np.int64)
        pick = rng.random(nwin)
        xs = np.where(pick < 0.08, 1, np.where(pick < 0.16, nxc - 2, xs))
        xs = np.clip(xs, 0, nxc - 1)
        r = y * nxc + xs
        kind = rng.random(nwin)
        f = foreign / 4
        r = np.where(kind < f, _abi.NO_MATCH, r)
        r = np.where((kind >= f) & (kind < 2 * f), (y + 1) * nxc + xs, r)
        r = np.where((kind >= 2 * f) & (kind < 3 * f), nxc * nyc + rng.integers(0, 1000, nwin), r)
        r = np.where((kind >= 3 * f) & (kind < 4 * f), 0xFFFFFFFE, r)
        out[i] = r
    return out.astype(np.uint32)


def refinable(shape, p, ri):
    """[n, nwin] bool: the target is a candidate of its window and both neighbours are too (the parabola is fitted)."""
    nx, ny, nxc, nyc, x, y, lo, hi = _geometry(shape, p)
    r = ri.astype(np.int64)
    xs = r % nxc
    cand = (r != _abi.NO_MATCH) & (r // nxc == y) & (xs >= lo) & (xs <= hi)
    return cand & (xs - 1 >= lo) & (xs + 1 <= hi)


def _round_half_away(t):
    a = abs(t)
    m = math.floor(a)
    return math.copysign(m + (1.0 if a - m >= 0.5 else 0.0), t)


def classify(left, right, p, ri):
    """The arm every window takes, from costs computed here (int64 SAD / SSD; NCC / ZNCC scored with the device's
    operations, test_gpu_limits._scores). Returns (arm [n, nwin], largest c(x*-1) + c(x*+1), largest 16 |num|,
    largest den) over the fitted windows of an integer cost (0 for NCC / ZNCC)."""
    n, h, w = left.shape[:3]
    c = left[0, 0].size // w
    nx, ny, nxc, nyc, x, y, lo, hi = _geometry(left.shape, p)
    tw, th, kind = p.tmpl_w, p.tmpl_h, p.cost_kind
    integer = kind <= _abi.COST_SSD
    arm = np.full(ri.shape, NONE, np.int64)
    sums = nums = dens = 0
    for i in range(n):
        L = left[i].reshape(h, w * c).astype(np.int64)
        R = right[i].reshape(h, w * c).astype(np.int64)
        for k in range(nx * ny):
            r = int(ri[i, k])
            xs = r % nxc
            if r == _abi.NO_MATCH or r // nxc != y[k] or not lo[k] <= xs <= hi[k]:
                continue
            if xs - 1 < lo[k] or xs + 1 > hi[k]:
                arm[i, k] = EDGE
                continue
            t = L[y[k]:y[k] + th, x[k] * c:(x[k] + tw) * c].ravel()
            b = np.stack([R[y[k]:y[k] + th, j * c:(j + tw) * c].ravel() for j in (xs - 1, xs, xs + 1)])
            if integer:
                cm, c0, cp = (np.abs(b - t).sum(1) if kind == _abi.COST_SAD else ((b - t) ** 2).sum(1)).tolist()
                num, den = cm - cp, cm + cp - 2 * c0
                sums, nums, dens = max(sums, cm + cp), max(nums, 16 * abs(num)), max(dens, den)
                if den == 0:
                    arm[i, k] = DEN0
                elif den < 0:
                    arm[i, k] = DENNEG
                else:
                    m = (16 * abs(num) + den) // (2 * den)
                    arm[i, k] = FIT if m <= 8 else CLAMP_P if num > 0 else CLAMP_M
            else:
                ones = np.ones(3, np.int64)
                sc = _scores(kind, t.size, (b * t).sum(1), ones * t.sum(), b.sum(1), ones * (t * t).sum(), (b * b).sum(1))
                vm, v0, vp = (1.0 - sc).tolist()
                num, den = vm - vp, (vm - v0) + (vp - v0)
                if den == 0:
                    arm[i, k] = DEN0
                elif den < 0:
                    arm[i, k] = DENNEG
                else:
                    q = _round_half_away(8.0 * num / den)
                    arm[i, k] = FIT if abs(q) <= 8 else CLAMP_P if q > 0 else CLAMP_M
    return arm, sums, nums, dens


def arm_counts(arm):
    return {ARM_NAMES[a]: int((arm == a).sum()) for a in range(7)}


# ---- the arm frames: small frames whose costs have known shapes -----------------------------------------------------
ARM_W, ARM_H, ARM_TW, ARM_TH = 40, 8, 5, 3
ARM_RANGES = {"signed": (-6, 6), "clipped": (3, 14), "bounded": (0, 9), "unbounded": (0, UNBOUNDED)}


def arm_frames(kind, c, seed):
    """ramp: a horizontal ramp, so SSD is a parabola in x' (every target one pixel or more from its vertex is clamped)
    and SAD is linear (collinear costs, den = 0); wave: a sinusoid of period 7, whose cost maxima give den < 0;
    texture: synthetic noise (fitted and clamped windows of every cost); full: both frames 255 (NCC / ZNCC tie
    everywhere, den = 0)."""
    shape = (1, ARM_H, ARM_W + 3, c)
    xx = np.arange(ARM_W + 3)[None, None, :, None]
    ch = np.arange(c)[None, None, None, :]
    if kind == "texture":
        l, r = synth.make_pairs(1, ARM_W, ARM_H, c, shift=3, noise_sigma=2.0, seed=seed)
        return np.ascontiguousarray(l), np.ascontiguousarray(r)
    if kind == "full":
        world = np.full(shape, 255, np.uint8)
    elif kind == "ramp":
        world = np.broadcast_to(np.clip(4 * xx + 9 * ch + 3, 0, 255), shape).astype(np.uint8)
    else:
        world = np.broadcast_to(np.rint(128 + 100 * np.sin(2 * np.pi * xx / 7 + ch)), shape).astype(np.uint8)
    l, r = world[:, :, 2:2 + ARM_W], world[:, :, :ARM_W]
    if c == 1:
        l, r = l[..., 0], r[..., 0]
    return np.ascontiguousarray(l), np.ascontiguousarray(r)


def arm_cases(cost, side, c):
    """(name, left, right, params, right_index) of every arm frame at every range, with `targets`."""
    rng = np.random.default_rng(100 * c + side)
    for kind in ("ramp", "wave", "texture", "full"):
        left, right = arm_frames(kind, c, seed=c)
        for rname, (dmin, dmax) in ARM_RANGES.items():
            p = _abi.make_params(tmpl_w=ARM_TW, tmpl_h=ARM_TH, cost=cost, camera_side=side, search_min=dmin, search_max=dmax,
                                 distance_kind=_abi.DIST_POWERLAW if rname == "clipped" else _abi.DIST_PINHOLE)
            yield "%s/%s" % (kind, rname), left, right, p, targets(left.shape, p, rng)


def _assert_every_arm(counts, what):
    assert all(v > 0 for v in counts.values()), "%s: an arm was not reached: %s" % (what, counts)


# ---- CPU: the oracle on caller-chosen targets -----------------------------------------------------------------------
@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("side", SIDES)
@pytest.mark.parametrize("cost", COSTS)
def test_oracle_on_caller_targets(oracle, sub, cost, side, c):
    arm_all = []
    for name, left, right, p, ri in arm_cases(cost, side, c):
        x16, dist = sub.refine_subpixel(left, right, p, ri)
        assert np.array_equal(x16, restate(oracle, left, right, p, ri)), name
        arm = classify(left, right, p, ri)[0]
        assert np.array_equal(x16 == _abi.NO_SUBPIXEL, arm == NONE), name
        frac = x16.astype(np.int64) - 16 * ((x16.astype(np.int64) + 8) // 16)  # +-q in [-8, 7]: q = +-8 reads as -8
        assert (np.abs(frac[(arm == CLAMP_P) | (arm == CLAMP_M)]) == 8).all(), name
        assert (frac[(arm == EDGE) | (arm == DEN0) | (arm == DENNEG)] == 0).all(), name
        assert (dist[arm == NONE] == 0.0).all()
        arm_all.append(arm.ravel())
    _assert_every_arm(arm_counts(np.concatenate(arm_all)), "%s side=%d c=%d" % (cost, side, c))


def test_targets_reach_the_row_ends():
    """`targets` hands the kernel x* = 1 and x* = nxc - 2 as fitted candidates (the loads that end at the first and the
    last byte of the row), and every kind of non-candidate."""
    left = np.zeros((1, 12, 37, 3), np.uint8)
    p = _abi.make_params(tmpl_w=6, tmpl_h=4, search_min=-UNBOUNDED, search_max=UNBOUNDED)
    ri = targets(left.shape, p, np.random.default_rng(0))
    nxc, nyc = 32, 9
    fit = refinable(left.shape, p, ri)
    assert fit[ri % nxc == 1].any() and fit[ri % nxc == nxc - 2].any()
    assert (ri == _abi.NO_MATCH).any() and (ri == 0xFFFFFFFE).any()
    assert ((ri >= nxc * nyc) & (ri < nxc * nyc + 1000)).any()


# ---- GPU helpers ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def device_frames(torch, frames, pad=16, gap=0, fill=0, rng=None):
    """frames [n, H, W(, C)] into one device buffer: rows 16-byte aligned with at least `pad` bytes of padding, `gap`
    bytes (a multiple of 16) between frames, padding and gaps holding `fill` (a byte, or "random").
    Returns (tensor, FrameDesc)."""
    n, h, w = frames.shape[:3]
    rb = frames[0, 0].size
    c = rb // w
    row_stride = (rb + pad + 15) & ~15
    frame_stride = h * row_stride + gap
    total = n * frame_stride
    buf = rng.integers(0, 256, total, dtype=np.uint8) if fill == "random" else np.full(total, fill, np.uint8)
    view = np.lib.stride_tricks.as_strided(buf, shape=(n, h, rb), strides=(frame_stride, row_stride, 1))
    view[...] = np.ascontiguousarray(frames).reshape(n, h, rb)
    return torch.from_numpy(buf).cuda(), _abi.FrameDesc(w, h, c, row_stride, frame_stride)


def refine_on_device(ctx, dl, dr, f, n, p, ri, want=("x16", "dist")):
    """usv_refine_subpixel_device on device frames and the RightIndex `ri` [n, nwin]; the outputs start as sentinels.
    Returns (x16, dist), None for an output not asked for."""
    torch = pytest.importorskip("torch")
    nwin = ri.shape[1]
    d_ri = torch.from_numpy(np.ascontiguousarray(ri, np.uint32).view(np.int32).ravel()).cuda()
    x16 = torch.full((n * nwin,), X16_SENTINEL, dtype=torch.int32, device="cuda") if "x16" in want else None
    dist = torch.full((n * nwin,), DIST_SENTINEL, dtype=torch.float64, device="cuda") if "dist" in want else None
    launches = ctx.launch_count
    stream = torch.cuda.current_stream().cuda_stream
    ctx.refine_subpixel_device(dl.data_ptr(), dr.data_ptr(), f, n, p, d_ri.data_ptr(), x16.data_ptr() if x16 is not None else None,
                               dist.data_ptr() if dist is not None else None, stream)
    torch.cuda.synchronize()
    assert api.lib().usv_device_status(ctx._h) == 0
    assert ctx.launch_count == launches + 1
    return (x16.cpu().numpy().reshape(n, nwin) if x16 is not None else None,
            dist.cpu().numpy().reshape(n, nwin) if dist is not None else None)


def refine_frames(ctx, left, right, p, ri, pad=16, gap=0, fill=0, seed=0, want=("x16", "dist")):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(seed)
    dl, f = device_frames(torch, left, pad, gap, fill, rng)
    dr, _ = device_frames(torch, right, pad, gap, fill, rng)
    return refine_on_device(ctx, dl, dr, f, left.shape[0], p, ri, want)


def check_vs_oracle(sub, left, right, p, ri, x16, dist, what=""):
    """The device's outputs against the oracle's (either may be None). Returns the oracle's disparity_x16."""
    ex16, edist = sub.refine_subpixel(left, right, p, ri)
    if x16 is not None:
        bad = np.nonzero(x16 != ex16)
        assert len(bad[0]) == 0, "%s: %d mismatches, first at (pair, window) %s: got %s expected %s (targets %s)" % (
            what, len(bad[0]), list(zip(bad[0][:3], bad[1][:3])), x16[bad][:3], ex16[bad][:3], ri[bad][:3])
    if dist is not None:
        if p.distance_kind == _abi.DIST_POWERLAW:
            assert np.array_equal(dist == 0, edist == 0) and np.array_equal(np.isnan(dist), np.isnan(edist)), what
            assert np.allclose(dist, edist, rtol=1e-12, atol=0, equal_nan=True), what
        else:  # PINHOLE: IEEE divisions and products; NONE: 0.0
            assert dist.tobytes() == edist.tobytes(), what
    return ex16


# ---- GPU: the caller-chosen targets through the device ----------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("cost", COSTS)
def test_device_on_caller_targets(ctx, sub, cost, c):
    for side in SIDES:
        arm_all = []
        for name, left, right, p, ri in arm_cases(cost, side, c):
            x16, dist = refine_frames(ctx, left, right, p, ri, fill="random", seed=c)
            check_vs_oracle(sub, left, right, p, ri, x16, dist, "%s side=%d" % (name, side))
            arm_all.append(classify(left, right, p, ri)[0].ravel())
        _assert_every_arm(arm_counts(np.concatenate(arm_all)), "%s side=%d c=%d" % (cost, side, c))


# ---- GPU: the integer limits ------------------------------------------------------------------------------------------
# 32768-byte templates at every channel count (10 x 1092 x 3 = 32760)
BIG = {1: (32, 1024), 2: (16, 1024), 3: (10, 1092), 4: (8, 1024)}
BIG_SHIFT = 5


def big_frames(kind, c, side, seed):
    """[1, th + 2, tw + 40(, C)] frames for the largest template. saturated: left 255 / right 0, every candidate costs
    the maximum; zero_cols / full_cols: a 0 (255) left frame against a 255 right frame with a 0 column every 13 pixels
    (costs near the maximum that step with the columns); random_cols: random 0 / 255 columns and the right frame
    shifted by BIG_SHIFT, so a target next to the match has one neighbour at cost 0 and the others near half the
    maximum (16 |num| near 8 * 65025 * 32768, den near 0 with either sign); flip_cols: the same with neighbouring columns
    unequal 3 times in 4, so a target on the match has den near 1.5 times the maximum; full and dips as in
    test_gpu_limits."""
    tw, th = BIG[c]
    h, w = th + 2, tw + 40
    shape = (1, h, w) if c == 1 else (1, h, w, c)
    if kind in ("saturated", "full", "dips"):
        return pattern(kind, 1, h, w, c, camera_side=side, seed=seed)
    if kind in ("zero_cols", "full_cols"):
        col = np.where(np.arange(w) % 13 == 0, 0, 255).astype(np.uint8)
        right = np.ascontiguousarray(np.broadcast_to(col[:, None], (w, c)).reshape(w * c)[None, None, :].repeat(h, 1).reshape(shape))
        left = np.full(shape, 0 if kind == "zero_cols" else 255, np.uint8)
        return left, right
    rng = np.random.default_rng(seed)
    if kind == "random_cols":
        cols = np.where(rng.random((w + BIG_SHIFT, c)) < 0.5, 0, 255).astype(np.uint8)
    else:  # flip_cols: each byte column differs from the one a pixel to its left with probability 3/4
        flips = rng.random((w + BIG_SHIFT, c)) < 0.75
        cols = np.where(np.cumsum(flips, axis=0) % 2 == 1, 255, 0).astype(np.uint8)
    world = np.ascontiguousarray(np.broadcast_to(cols[None], (h, w + BIG_SHIFT, c)))[None]
    a, b = world[:, :, :w], world[:, :, BIG_SHIFT:BIG_SHIFT + w]
    left, right = (a, b) if side == _abi.LEFT_CAM else (b, a)
    return np.ascontiguousarray(left.reshape(shape)), np.ascontiguousarray(right.reshape(shape))


BIG_KINDS = {"ssd": ("saturated", "zero_cols", "full_cols", "random_cols", "flip_cols"), "sad": ("saturated", "full", "dips", "random_cols"),
             "ncc": ("saturated", "full", "dips", "random_cols"), "zncc": ("saturated", "full", "dips", "random_cols")}


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("cost", COSTS)
def test_largest_template(ctx, sub, cost, c):
    tw, th = BIG[c]
    assert tw * th * c in (32768, 32760)
    rng = np.random.default_rng(c)
    sums = nums = dens = 0
    arm_all = []
    for side in SIDES:
        for kind in BIG_KINDS[cost]:
            left, right = big_frames(kind, c, side, seed=c + side)
            p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost=cost, camera_side=side, search_min=0, search_max=2 * BIG_SHIFT)
            ri = targets(left.shape, p, rng, foreign=0.05)
            x16, dist = refine_frames(ctx, left, right, p, ri, fill="random", seed=c)
            check_vs_oracle(sub, left, right, p, ri, x16, dist, "%s side=%d" % (kind, side))
            arm, s, n16, d = classify(left, right, p, ri)
            sums, nums, dens = max(sums, s), max(nums, n16), max(dens, d)
            arm_all.append(arm.ravel())
    counts = arm_counts(np.concatenate(arm_all))
    assert counts[ARM_NAMES[DEN0]] > 0 and counts[ARM_NAMES[FIT]] > 0, counts
    if cost == "ssd":
        # past the 32-bit signed range in every intermediate of the int64 arm: c(x*-1) + c(x*+1) and den beyond 2^31
        # (the sum of two costs stays below 2^32), 16 |num| beyond 2^32
        assert sums > 2 ** 31 and dens > 2 ** 31 and nums > 2 ** 32, (sums, dens, nums)
        assert counts[ARM_NAMES[CLAMP_P]] > 0 and counts[ARM_NAMES[CLAMP_M]] > 0, counts


# ---- GPU: geometry ----------------------------------------------------------------------------------------------------
# name: (channels, width, height, tmpl_w, tmpl_h, stride_x, stride_y, n_pairs, gap)
GEOMS = {
    # every residue of tw*C mod 4 the channel count allows, on widths whose rows end inside a word
    "res_c1": (1, 45, 12, [4, 5, 6, 7], 3, 1, 1, 1, 0),
    "res_c2": (2, 43, 12, [2, 3], 3, 1, 1, 1, 0),
    "res_c3": (3, 41, 12, [4, 1, 2, 3], 3, 1, 1, 1, 0),
    "res_c4": (4, 39, 12, [1, 3], 3, 1, 1, 1, 0),
    # one template word per row (the word loop does not run), and one-row templates
    "one_word_c1": (1, 29, 9, [1, 2, 3], 1, 1, 1, 1, 0),
    "one_word_c2": (2, 29, 9, [1], 2, 1, 1, 1, 0),
    "one_word_c3": (3, 29, 9, [1], 4, 1, 1, 1, 0),
    "one_word_c4": (4, 29, 9, [1], 5, 1, 1, 1, 0),
    "th1": (3, 33, 7, [9], 1, 1, 1, 1, 0),
    # 1024-byte template rows (1023 at C = 3)
    "row1024_c1": (1, 1061, 8, [1024], 3, 1, 1, 1, 0),
    "row1024_c2": (2, 549, 8, [512], 4, 1, 1, 1, 0),
    "row1024_c3": (3, 375, 8, [341], 2, 1, 1, 1, 0),
    "row1024_c4": (4, 293, 8, [256], 5, 1, 1, 1, 0),
    # more than one 128-window CTA per row, not a multiple of 128, with strides 1 to 3
    "wide_s1": (1, 301, 10, [7], 4, 1, 1, 1, 0),
    "wide_s2_c3": (3, 547, 10, [6], 3, 2, 3, 1, 0),
    "wide_s3_c2": (2, 811, 14, [5], 2, 3, 2, 1, 0),
    # three distinct pairs with a gap between frames
    "pairs3_c1": (1, 157, 20, [9], 7, 1, 1, 3, 48),
    "pairs3_c4": (4, 61, 20, [5], 3, 2, 1, 3, 4096),
    "pairs3_c3": (3, 97, 20, [11], 5, 3, 3, 3, 16),
}


def _geom_frames(c, w, h, n, seed):
    left, right = synth.make_pairs(n, w, h, c, shift=6, noise_sigma=2.0, seed=seed)
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    left[:, :, :3] = 90  # a flat block: ties, zero variance
    right[:, :, :3] = 90
    return left, right


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GEOMS))
def test_geometry(ctx, sub, name):
    c, w, h, tws, th, sx, sy, n, gap = GEOMS[name]
    assert (w * c) % 4 != 0 or c == 4
    left, right = _geom_frames(c, w, h, n, seed=w)
    rng = np.random.default_rng(w)
    ends = [0, 0]
    fractional = 0
    for tw in tws:
        for k, cost in enumerate(COSTS):
            for side in SIDES:
                # the whole row is the range: x* = 1 and x* = nxc - 2 are fitted for every window
                rng_kind = (k + side) % 3
                dmin, dmax = ((-UNBOUNDED, UNBOUNDED), (-7, 7), (0, UNBOUNDED))[rng_kind]
                p = _abi.make_params(tmpl_w=tw, tmpl_h=th, stride_x=sx, stride_y=sy, cost=cost, camera_side=side, search_min=dmin,
                                     search_max=dmax, distance_kind=(_abi.DIST_PINHOLE, _abi.DIST_POWERLAW)[k % 2])
                ri = targets(left.shape, p, rng)
                fill = (0xFF, "random")[k % 2]
                x16, dist = refine_frames(ctx, left, right, p, ri, gap=gap, fill=fill, seed=k)
                ex16 = check_vs_oracle(sub, left, right, p, ri, x16, dist, "tw=%d %s side=%d fill=%s" % (tw, cost, side, fill))
                nxc = w - tw + 1
                fit = refinable(left.shape, p, ri)
                if rng_kind == 0:
                    ends[0] += int((fit & (ri % nxc == 1)).sum())
                    ends[1] += int((fit & (ri % nxc == nxc - 2)).sum())
                fractional += int((ex16[fit] % 16 != 0).sum())
    assert ends[0] > 0 and ends[1] > 0 and fractional > 0, (ends, fractional)


@pytest.mark.gpu
def test_more_than_65535_window_rows(ctx, sub):
    """A 12-px gray frame 65 543 rows tall with a 4x4 template: 65 540 window rows, so the grid holds 65 535 and the
    kernel's row loop takes a second turn for the last five."""
    h, w = 65543, 12
    rng = np.random.default_rng(65543)
    left = rng.integers(0, 256, (1, h, w), dtype=np.uint8)
    right = np.ascontiguousarray(np.roll(left, -2, axis=2))
    torch = pytest.importorskip("torch")
    dl, f = device_frames(torch, left, fill="random", rng=rng)
    dr, _ = device_frames(torch, right, fill="random", rng=rng)
    for cost in COSTS:
        p = _abi.make_params(tmpl_w=4, tmpl_h=4, cost=cost, search_min=-4, search_max=4, distance_kind=_abi.DIST_POWERLAW)
        nx, ny = api.grid_dims(f, p)[:2]
        assert ny == 65540 > 65535
        ri = targets(left.shape, p, rng)
        x16, dist = refine_on_device(ctx, dl, dr, f, 1, p, ri)
        ex16 = check_vs_oracle(sub, left, right, p, ri, x16, dist, cost)
        tail = ex16[0, 65535 * nx:]
        assert (tail != _abi.NO_SUBPIXEL).sum() > 0 and (tail % 16 != 0).any()


# ---- GPU: output pointers and the host entry point ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 2, 3, 4])
def test_each_output_alone(ctx, sub, c):
    """disparity_x16 alone and distance alone are what the run with both writes; DIST_NONE writes 0.0 distances."""
    left, right = _geom_frames(c, 77, 16, 2, seed=c)
    rng = np.random.default_rng(c)
    for k, cost in enumerate(COSTS):
        for dist_kind in (_abi.DIST_NONE, _abi.DIST_PINHOLE, _abi.DIST_POWERLAW):
            p = _abi.make_params(tmpl_w=7, tmpl_h=5, stride_x=1 + k % 2, cost=cost, camera_side=SIDES[k % 2], search_min=-3,
                                 search_max=20, distance_kind=dist_kind)
            ri = targets(left.shape, p, rng)
            both = refine_frames(ctx, left, right, p, ri, gap=32)
            ex16 = check_vs_oracle(sub, left, right, p, ri, *both, what="%s dist=%d" % (cost, dist_kind))
            x16_only = refine_frames(ctx, left, right, p, ri, gap=32, want=("x16",))
            dist_only = refine_frames(ctx, left, right, p, ri, gap=32, want=("dist",))
            assert x16_only[1] is None and dist_only[0] is None
            assert x16_only[0].tobytes() == both[0].tobytes() and dist_only[1].tobytes() == both[1].tobytes()
            if dist_kind == _abi.DIST_NONE:
                assert (both[1] == 0.0).all() and (ex16 != _abi.NO_SUBPIXEL).any()


def _odd_stride_batch(frames, extra, gap):
    """frames [n, H, W, C] as a view into a host buffer whose rows are W*C + extra bytes apart (odd) and whose frames
    are `gap` bytes further apart than that."""
    n, h = frames.shape[:2]
    rb = frames[0, 0].size
    rs = rb + extra
    fs = h * rs + gap
    buf = np.full(n * fs, 0xA5, np.uint8)
    view = np.lib.stride_tricks.as_strided(buf, shape=frames.shape, strides=(fs, rs) + frames.strides[2:])
    view[...] = frames
    return buf, view


@pytest.mark.gpu
@pytest.mark.parametrize("c", [2, 4])
def test_host_entry(ctx, sub, oracle, c):
    """usv_match_dense_subpixel_host at C = 2 and 4 (always the direct form), strided grids, an odd host row stride
    (the frames are repacked on their way to the device) and three pairs with a gap between frames."""
    left, right = _geom_frames(c, 67, 23, 3, seed=10 + c)
    _, lv = _odd_stride_batch(left, 2 * c + 1, 7)
    _, rv = _odd_stride_batch(right, 2 * c + 1, 7)
    assert lv.strides[1] % 2 == 1 and lv.strides[0] > lv.strides[1] * lv.shape[1]
    for k, cost in enumerate(COSTS):
        p = _abi.make_params(tmpl_w=(5, 6, 7, 3)[k], tmpl_h=4, stride_x=1 + k % 3, stride_y=1 + (k + 1) % 3, cost=cost,
                             camera_side=SIDES[k % 2], search_min=-4, search_max=30,
                             distance_kind=(_abi.DIST_PINHOLE, _abi.DIST_POWERLAW)[k % 2])
        got = ctx.match_dense_subpixel(lv, rv, p, mask=_abi.OUT_RIGHT_INDEX)
        assert ctx.last_kernel == "block_cost_argmin_direct"
        ri = got["right_index"]
        assert ri.shape[0] == 3 and (ri != _abi.NO_MATCH).any()
        assert np.array_equal(ri, oracle.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX)["right_index"])
        check_vs_oracle(sub, left, right, p, ri, got["disparity_x16"], got["subpixel_distance"], cost)


# ---- GPU: all 16 instances behind the sweep that serves them -----------------------------------------------------------
# (cost, channels, tmpl_w, tmpl_h, stride, corr kernel option, expected sweep kernel)
INSTANCES = [
    ("sad", 1, 12, 7, 1, "auto", "dense_sad_argmin_kernel"),
    ("ssd", 1, 13, 9, 1, "auto", "dense_corr_mma_kernel"),
    ("ncc", 1, 11, 6, 1, "auto", "dense_corr_umma_kernel"),
    ("zncc", 1, 16, 5, 1, "alu", "dense_corr_argmin_kernel"),
    ("sad", 3, 8, 6, 1, "auto", "dense_sad_argmin_kernel"),
    ("ssd", 3, 7, 5, 1, "auto", "dense_corr_mma_kernel"),
    ("ncc", 3, 13, 4, 1, "auto", "dense_corr_mma_kernel"),
    ("zncc", 3, 24, 3, 1, "alu", "dense_corr_argmin_kernel"),
    ("sad", 2, 9, 5, 2, "auto", "block_cost_argmin_direct"),
    ("ssd", 2, 6, 7, 1, "auto", "block_cost_argmin_direct"),
    ("ncc", 2, 11, 3, 3, "auto", "block_cost_argmin_direct"),
    ("zncc", 2, 4, 8, 1, "auto", "block_cost_argmin_direct"),
    ("sad", 4, 5, 6, 1, "auto", "block_cost_argmin_direct"),
    ("ssd", 4, 3, 4, 2, "auto", "block_cost_argmin_direct"),
    ("ncc", 4, 8, 3, 3, "auto", "block_cost_argmin_direct"),
    ("zncc", 4, 6, 5, 1, "auto", "block_cost_argmin_direct"),
]


def sweep_on_device(ctx, dl, dr, f, n, p, kernel="auto"):
    """usv_match_dense_device with RightIndex into HBM: (right_index [n, nwin], usv_last_kernel)."""
    torch = pytest.importorskip("torch")
    nx, ny, _ = api.grid_dims(f, p)
    ri = torch.zeros(n * nx * ny, dtype=torch.int32, device="cuda")
    st = _abi.Outputs()
    st.right_index = ri.data_ptr()
    ctx.corr_kernel(kernel)
    try:
        ctx.match_dense_device(dl.data_ptr(), dr.data_ptr(), f, n, p, st, torch.cuda.current_stream().cuda_stream)
    finally:
        ctx.corr_kernel("auto")
    torch.cuda.synchronize()
    assert api.lib().usv_device_status(ctx._h) == 0
    return ri.cpu().numpy().view(np.uint32).reshape(n, nx * ny), ctx.last_kernel


@pytest.mark.gpu
@pytest.mark.parametrize("inst", INSTANCES, ids=lambda t: "%s-c%d-%s" % (t[0], t[1], t[6]))
def test_every_instance_behind_its_sweep(ctx, sub, inst):
    torch = pytest.importorskip("torch")
    cost, c, tw, th, s, kernel, expect = inst
    for side in SIDES:
        left, right = synth.make_pairs(2, 157, 30, c, shift=11 if side == _abi.LEFT_CAM else -11, noise_sigma=2.0, seed=c + tw)
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        rng = np.random.default_rng(tw)
        dl, f = device_frames(torch, left, gap=64, fill="random", rng=rng)
        dr, _ = device_frames(torch, right, gap=64, fill="random", rng=rng)
        # a signed range: candidates on both sides of the window
        p = _abi.make_params(tmpl_w=tw, tmpl_h=th, stride_x=s, stride_y=1 + (s - 1) // 2, cost=cost, camera_side=side, search_min=-5,
                             search_max=40, accept_threshold=3.0, distance_kind=(_abi.DIST_PINHOLE, _abi.DIST_POWERLAW)[side])
        ri, name = sweep_on_device(ctx, dl, dr, f, 2, p, kernel)
        assert name == expect
        assert (ri != _abi.NO_MATCH).all()
        x16, dist = refine_on_device(ctx, dl, dr, f, 2, p, ri)
        assert ctx.last_kernel == name
        ex16 = check_vs_oracle(sub, left, right, p, ri, x16, dist, "side=%d" % side)
        assert (ex16 % 16 != 0).any()


# ---- GPU: seeded random configurations --------------------------------------------------------------------------------
def random_config(seed):
    rng = np.random.default_rng(seed)
    cost = COSTS[rng.integers(4)]
    c = int(rng.integers(1, 5))
    tw, th = int(rng.integers(1, 65)), int(rng.integers(1, 41))
    w = tw + int(rng.integers(3, 90))
    if (w * c) % 4 == 0:
        w += 1
    h = th + int(rng.integers(0, 12))
    sx, sy = int(rng.integers(1, 4)), int(rng.integers(1, 4))
    rname = ("bounded", "signed", "clipped", "empty", "unbounded")[rng.integers(5)]
    a, b = int(rng.integers(0, 20)), int(rng.integers(0, 40))
    dmin, dmax = {"bounded": (0, a + b), "signed": (-a, b), "clipped": (a + 3, a + 3 + b), "empty": (w + 5, w + 50),
                  "unbounded": (0, UNBOUNDED)}[rname]
    side = SIDES[rng.integers(2)]
    n = int(rng.integers(1, 4))
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, stride_x=sx, stride_y=sy, cost=cost, camera_side=side, search_min=dmin,
                         search_max=dmax, accept_threshold=float(rng.choice([3.0, 0.5])),
                         distance_kind=int(rng.integers(0, 3)))
    cfg = dict(seed=seed, cost=cost, c=c, w=w, h=h, tw=tw, th=th, sx=sx, sy=sy, range=rname, search=(dmin, dmax),
               side=side, n=n, threshold=p.accept_threshold, distance_kind=p.distance_kind)
    return cfg, p, rng


def perturb(ri, shape, p, rng):
    """The sweep's winners with a share of perturbed targets: x* +- 1..3, a candidate of another row, NO_MATCH, past the
    frame."""
    nx, ny, nxc, nyc, x, y, lo, hi = _geometry(shape, p)
    r = ri.astype(np.int64)
    has = r != _abi.NO_MATCH
    xs, ys = np.where(has, r % nxc, x), np.where(has, r // nxc, y)
    kind = rng.integers(0, 10, r.shape)
    k = rng.integers(1, 4, r.shape) * rng.choice([-1, 1], r.shape)
    moved = ys * nxc + np.clip(xs + k, 0, nxc - 1)
    r = np.where(kind == 5, moved, r)
    r = np.where(kind == 6, np.where(ys + 1 < nyc, ys + 1, 0) * nxc + xs, r)
    r = np.where(kind == 7, _abi.NO_MATCH, r)
    r = np.where(kind == 8, nxc * nyc + rng.integers(0, 50, r.shape), r)
    r = np.where(kind == 9, y * nxc + np.clip(x + k, 0, nxc - 1), r)
    return r.astype(np.uint32)


@pytest.mark.gpu
def test_random_configurations(ctx, sub):
    torch = pytest.importorskip("torch")
    refined = fractional = none = 0
    kernels = set()
    for seed in range(100):
        cfg, p, rng = random_config(seed)
        left, right = synth.make_pairs(cfg["n"], cfg["w"], cfg["h"], cfg["c"], shift=int(rng.integers(-12, 13)), noise_sigma=2.0,
                                       seed=seed)
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        if rng.random() < 0.5:  # a flat region in both frames
            y0, x0 = int(rng.integers(0, cfg["h"])), int(rng.integers(0, cfg["w"]))
            v = int(rng.integers(0, 256))
            left[:, y0:y0 + 8, x0:x0 + 12], right[:, y0:y0 + 8, x0:x0 + 12] = v, v
        fill = ("random", 0xFF, 0)[seed % 3]
        dl, f = device_frames(torch, left, pad=int(rng.integers(0, 40)), gap=16 * int(rng.integers(0, 5)), fill=fill, rng=rng)
        dr, _ = device_frames(torch, right, pad=f.row_stride - left[0, 0].size, gap=f.frame_stride - f.row_stride * cfg["h"],
                              fill=fill, rng=rng)
        ri, name = sweep_on_device(ctx, dl, dr, f, cfg["n"], p)
        kernels.add(name)
        ri = perturb(ri, left.shape, p, rng)
        x16, dist = refine_on_device(ctx, dl, dr, f, cfg["n"], p, ri)
        ex16 = check_vs_oracle(sub, left, right, p, ri, x16, dist, "config %s" % cfg)
        refined += int((ex16 != _abi.NO_SUBPIXEL).sum())
        fractional += int(((ex16 != _abi.NO_SUBPIXEL) & (ex16 % 16 != 0)).sum())
        none += int((ex16 == _abi.NO_SUBPIXEL).sum())
    assert refined > 0 and fractional > 0 and none > 0
    assert "block_cost_argmin_direct" in kernels and len(kernels) > 1, kernels
