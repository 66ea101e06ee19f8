"""Sub-pixel disparity of the dense sweep's winners (include/usv_b200.h: usv_refine_subpixel_device,
usv_match_dense_subpixel_host).

The refinement oracle is tests/subpixel_oracle.c (the block-search oracle's cost functions plus the refinement),
compiled by the `sub` fixture.
CPU: that oracle against an independent restatement built from the block-search oracle's candidate rows, the accuracy the
refinement buys on a known fractional shift, and the int64 arm at 32768-byte SSD templates on saturated frames.
GPU: the kernel bit for bit against the oracle behind every sweep family, the host call against match_dense, the
invariants at full size, the guard against indices that are not candidates, dirty row padding and the refusals."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth

ACCEPT_ALL = 3.0  # every MatchValue (SAD/SSD <= 1, NCC/ZNCC <= 2) is accepted
COSTS = ("sad", "ssd", "ncc", "zncc")


# ---- the refinement oracle (tests/subpixel_oracle.c) -------------------------------------------------------------
class SubpixelOracle:
    """ctypes wrapper of tests/subpixel_oracle.c, compiled into a temporary directory (OpenMP, no FMA contraction)."""

    def __init__(self, so_path):
        self.L = C.CDLL(so_path)
        self.L.usv_subpixel_oracle_distance_f64.restype = C.c_double
        self.L.usv_subpixel_oracle_distance_f64.argtypes = [C.c_double, C.c_int32]

    def refine_subpixel(self, left, right, params, right_index):
        """right_index [n, ny*nx] -> (disparity_x16 int32, distance f64), both [n, ny*nx]."""
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        f = _abi.frame_desc_for(left)
        nx, ny, _ = api.grid_dims(f, params)
        n = left.shape[0]
        ri = np.ascontiguousarray(right_index, np.uint32).reshape(n, ny * nx)
        x16 = np.zeros((n, ny * nx), np.int32)
        dist = np.zeros((n, ny * nx), np.float64)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        rc = self.L.usv_subpixel_oracle_refine(ptr(left), ptr(right), C.byref(f), C.c_int32(n), C.byref(params), ptr(ri), ptr(x16),
                                               ptr(dist))
        assert rc == 0
        return x16, dist

    def distance_f64(self, disp, kind):
        return np.array([self.L.usv_subpixel_oracle_distance_f64(float(d), int(kind)) for d in np.asarray(disp).ravel()], np.float64)


@pytest.fixture(scope="module")
def sub(tmp_path_factory):
    here = os.path.dirname(os.path.abspath(__file__))
    so = str(tmp_path_factory.mktemp("subpixel_oracle") / "libusv_subpixel_oracle.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"  # as oracle/Makefile: the system compiler has OpenMP
    out = subprocess.run([cc, "-O3", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-o", so,
                          os.path.join(here, "subpixel_oracle.c"), "-lm"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return SubpixelOracle(so)


# ---- the restatement ------------------------------------------------------------------------------------------------
def _round_half_away(t):
    a = abs(t)
    m = math.floor(a)
    return math.copysign(m + (1.0 if a - m >= 0.5 else 0.0), t)


def _q(costs, integer):
    cm, c0, cp = costs
    if integer:
        cm, c0, cp = int(cm), int(c0), int(cp)  # Python ints: no overflow at any template size
        num, den = cm - cp, cm + cp - 2 * c0
        if den <= 0:
            return 0
        m = min((16 * abs(num) + den) // (2 * den), 8)
        return -m if num < 0 else m
    num, den = cm - cp, (cm - c0) + (cp - c0)
    if not den > 0:
        return 0
    return int(min(max(_round_half_away(8.0 * num / den), -8.0), 8.0))


def restate(oracle, left, right, p, right_index):
    """disparity_x16 [n, ny*nx] from the oracle's candidate rows (match_templates(rows=True)): c(x*-1), c(x*), c(x*+1)
    read straight from the row of each window."""
    f = _abi.frame_desc_for(left)
    nx, ny, _ = oracle.grid_dims(f, p)
    nxc = f.width - p.tmpl_w + 1
    w = np.arange(nx * ny)
    tx, ty = (w % nx) * p.stride_x, (w // nx) * p.stride_y
    rows = oracle.match_templates(left, right, tx, ty, p, mask=_abi.OUT_RIGHT_INDEX, rows=True)
    integer = p.cost_kind <= _abi.COST_SSD
    out = np.full(right_index.shape, _abi.NO_SUBPIXEL, np.int64)
    for i in range(left.shape[0]):
        for k in range(nx * ny):
            r = int(right_index[i, k])
            x, y = int(tx[k]), int(ty[k])
            if p.camera_side == _abi.LEFT_CAM:
                lo, hi = max(x - p.search_max, 0), min(x - p.search_min, nxc - 1)
            else:
                lo, hi = max(x + p.search_min, 0), min(x + p.search_max, nxc - 1)
            xs = r % nxc
            if r == _abi.NO_MATCH or r // nxc != y or not lo <= xs <= hi:
                continue
            d = x - xs if p.camera_side == _abi.LEFT_CAM else xs - x
            q = 0
            if xs - 1 >= lo and xs + 1 <= hi:
                row = rows["cost_rows"][i, k] if integer else 1.0 - rows["score_rows"][i, k]
                q = _q(row[xs - 1 - lo:xs + 2 - lo], integer)
            out[i, k] = 16 * d - q if p.camera_side == _abi.LEFT_CAM else 16 * d + q
    return out.astype(np.int32)


def _pinhole(x16):
    with np.errstate(divide="ignore"):  # disparity 0: +inf, as on the device
        return ((201.6 * 4) / ((x16 / 16.0) * 0.000043)) / 1000


def _check_distance(x16, dist, kind, sub):
    has = x16 != _abi.NO_SUBPIXEL
    assert (dist[~has] == 0.0).all()
    if kind == _abi.DIST_PINHOLE:
        assert dist[has].tobytes() == _pinhole(x16[has].astype(np.float64)).tobytes()
    else:
        assert dist[has].tobytes() == sub.distance_f64(x16[has] / 16.0, kind).tobytes()


# ---- CPU: oracle against the restatement ----------------------------------------------------------------------------
RANGES = {"full": dict(), "signed": dict(search_min=-9, search_max=9), "clipped": dict(search_min=3, search_max=20)}


@pytest.mark.parametrize("rng_name", sorted(RANGES))
@pytest.mark.parametrize("side", [_abi.LEFT_CAM, _abi.RIGHT_CAM])
@pytest.mark.parametrize("cost", COSTS)
def test_oracle_equals_restatement(oracle, sub, cost, side, rng_name):
    for c, (tw, th), (sx, sy), thr in ((1, (7, 5), (1, 1), ACCEPT_ALL), (3, (8, 4), (3, 2), ACCEPT_ALL), (1, (5, 3), (2, 1), 0.0)):
        left, right = synth.make_pairs(2, 61, 19, c, shift=7 if side == _abi.LEFT_CAM else -7, noise_sigma=2.0, seed=5 + c)
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        left[1, :9], right[1, :9] = 77, 77  # flat rows: every candidate ties, the first wins at its range's end
        p = _abi.make_params(tmpl_w=tw, tmpl_h=th, stride_x=sx, stride_y=sy, cost=cost, camera_side=side,
                             accept_threshold=thr, **RANGES[rng_name])
        ri = oracle.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX)["right_index"]
        x16, dist = sub.refine_subpixel(left, right, p, ri)
        assert np.array_equal(x16, restate(oracle, left, right, p, ri)), (c, tw, th)
        assert np.array_equal(x16 == _abi.NO_SUBPIXEL, ri == _abi.NO_MATCH)
        _check_distance(x16, dist, p.distance_kind, sub)
        if thr == 0.0:
            assert (x16 == _abi.NO_SUBPIXEL).all()


@pytest.mark.parametrize("cost", COSTS)
def test_oracle_ties_and_range_ends(oracle, sub, cost):
    """Columns repeated in pairs: a 1-pixel-wide template often ties with its right neighbour, q = +8 (the midpoint of
    the tied pair); winners at either end of a clipped range keep q = 0."""
    rng = np.random.default_rng(4)
    cols = rng.integers(0, 256, (1, 12, 40), dtype=np.uint8)
    right = np.ascontiguousarray(np.repeat(cols, 2, axis=2)[:, :, :64])
    left = np.ascontiguousarray(np.roll(right, 6, axis=2))
    p = _abi.make_params(tmpl_w=1, tmpl_h=3, cost=cost, search_min=2, search_max=10, accept_threshold=ACCEPT_ALL,
                         distance_kind=_abi.DIST_POWERLAW)
    ri = oracle.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX)["right_index"]
    x16, dist = sub.refine_subpixel(left, right, p, ri)
    assert np.array_equal(x16, restate(oracle, left, right, p, ri))
    _check_distance(x16, dist, p.distance_kind, sub)
    frac = (x16[x16 != _abi.NO_SUBPIXEL] % 16)
    assert (frac == 0).any() and (frac == 8).any()  # range ends (q = 0) and ties (q = +8)


# ---- CPU: accuracy on a known fractional shift ----------------------------------------------------------------------
def _shifted_texture(h, w, shift, seed):
    """A band-limited random texture T and T(x - shift), resampled exactly in the Fourier domain (period 2w)."""
    rng = np.random.default_rng(seed)
    W = 2 * w
    spec = rng.normal(size=(h, W // 2 + 1)) + 1j * rng.normal(size=(h, W // 2 + 1))
    k = np.arange(W // 2 + 1)
    spec[:, k > W // 6] = 0  # below a third of the Nyquist frequency
    spec[:, 0] = 0
    a = np.fft.irfft(spec, W, axis=1)
    b = np.fft.irfft(spec * np.exp(-2j * np.pi * k * shift / W), W, axis=1)
    s = 90.0 / np.abs(a).max()
    to8 = lambda v: np.clip(np.rint(128 + s * v[:, :w]), 0, 255).astype(np.uint8)  # noqa: E731
    return to8(a), to8(b)


@pytest.mark.parametrize("cost", COSTS)
def test_subpixel_beats_integer_on_fractional_shift(oracle, sub, cost):
    for f in (0.25, 0.5, 0.75):
        true = 20 + f
        t, ts = _shifted_texture(24, 120, true, seed=int(f * 100))
        # right(x) = T(x - true): the left window at x is seen at x' = x + true, RightCam disparity `true`
        left, right = t[None], ts[None]
        p = _abi.make_params(tmpl_w=9, tmpl_h=9, cost=cost, camera_side=_abi.RIGHT_CAM, search_min=12, search_max=30,
                             accept_threshold=ACCEPT_ALL)
        out = oracle.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_DISPARITY_U16)
        x16, _ = sub.refine_subpixel(left, right, p, out["right_index"])
        nxc = 120 - 9 + 1
        ok = (out["right_index"] != _abi.NO_MATCH) & ((np.arange(x16.shape[1]) % nxc) + 30 < nxc)  # the shift is in view
        err_int = np.abs(out["disparity_u16"][ok].astype(np.float64) - true).mean()
        err_sub = np.abs(x16[ok] / 16.0 - true).mean()
        assert err_sub < err_int, (f, err_sub, err_int)


# ---- CPU: the int64 arm at the largest template ---------------------------------------------------------------------
def test_int64_arm_at_32768_byte_ssd(oracle, sub):
    """Saturated frames at a 32x1024 SSD template: a 0 frame against 255 with a 0 column every 13 pixels, and a 255
    frame against the same. Costs come near 65025 * 32768 and c(x*-1) + c(x*+1) passes 2^31."""
    h, w, tw, th = 1026, 44, 32, 1024
    col = np.where(np.arange(w) % 13 == 0, 0, 255).astype(np.uint8)
    right = np.ascontiguousarray(np.broadcast_to(col, (1, h, w)))
    for lval in (0, 255):
        left = np.full((1, h, w), lval, np.uint8)
        p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="ssd", search_min=-6, search_max=6, accept_threshold=ACCEPT_ALL)
        f = _abi.frame_desc_for(left)
        nx, ny, _ = oracle.grid_dims(f, p)
        nxc = w - tw + 1
        w_idx = np.arange(nx * ny)
        x, y = w_idx % nx, w_idx // nx
        xs = np.clip(x + (w_idx % 5) - 2, 1, nxc - 2)  # caller-chosen targets, inside the range and the frame
        ri = (y * nxc + xs).astype(np.uint32)[None]
        x16, _ = sub.refine_subpixel(left, right, p, ri)
        L, R = left[0].astype(np.int64), right[0].astype(np.int64)
        exp, sums = [], []
        for k in range(nx * ny):
            cs = [int(((L[y[k]:y[k] + th, x[k]:x[k] + tw] - R[y[k]:y[k] + th, j:j + tw]) ** 2).sum()) for j in (xs[k] - 1, xs[k], xs[k] + 1)]
            sums.append(cs[0] + cs[2])
            exp.append(16 * (int(x[k]) - int(xs[k])) - _q(cs, True))
        assert np.array_equal(x16[0], np.array(exp, np.int32))
        assert lval == 255 or max(sums) > 2 ** 31
        assert (x16[0] % 16 != 0).any()


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _device_frames(torch, frames, pad=16, fill=0, rng=None):
    """frames [n, H, W(, C)] into a device buffer with 16-byte aligned rows and `pad` bytes of padding per row holding
    `fill` (a byte, or "random"). Returns (tensor, FrameDesc)."""
    n, h, w = frames.shape[:3]
    c = frames.shape[3] if frames.ndim == 4 else 1
    pitch = (w * c + pad + 15) & ~15
    if fill == "random":
        buf = rng.integers(0, 256, (n, h, pitch), dtype=np.uint8)
    else:
        buf = np.full((n, h, pitch), fill, np.uint8)
    buf[:, :, :w * c] = np.ascontiguousarray(frames).reshape(n, h, w * c)
    return torch.from_numpy(buf).cuda(), _abi.FrameDesc(w, h, c, pitch, pitch * h)


def _sweep_and_refine(ctx, left, right, p, kernel="auto", fill=0, seed=0, ri_override=None):
    """Dense sweep on the device (RightIndex into HBM), then usv_refine_subpixel_device on it. Returns
    (right_index, disparity_x16, distance, disparity_u16, last_kernel) as [n, ny*nx] arrays."""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(seed)
    dl, f = _device_frames(torch, left, fill=fill, rng=rng)
    dr, _ = _device_frames(torch, right, fill=fill, rng=rng)
    n = left.shape[0]
    nx, ny, _ = api.grid_dims(f, p)
    nw = n * nx * ny
    ri = torch.zeros(nw, dtype=torch.int32, device="cuda")
    du = torch.zeros(nw, dtype=torch.int16, device="cuda")
    st = _abi.Outputs()
    st.right_index, st.disparity_u16 = ri.data_ptr(), du.data_ptr()
    stream = torch.cuda.current_stream().cuda_stream
    ctx.corr_kernel(kernel)
    try:
        ctx.match_dense_device(dl.data_ptr(), dr.data_ptr(), f, n, p, st, stream)
    finally:
        ctx.corr_kernel("auto")
    name = ctx.last_kernel
    if ri_override is not None:
        ri = torch.from_numpy(np.ascontiguousarray(ri_override, np.uint32).view(np.int32).ravel()).cuda()
    x16 = torch.zeros(nw, dtype=torch.int32, device="cuda")
    dist = torch.zeros(nw, dtype=torch.float64, device="cuda")
    launches = ctx.launch_count
    ctx.refine_subpixel_device(dl.data_ptr(), dr.data_ptr(), f, n, p, ri.data_ptr(), x16.data_ptr(), dist.data_ptr(), stream)
    torch.cuda.synchronize()
    assert api.lib().usv_device_status(ctx._h) == 0
    assert ctx.launch_count == launches + 1 and ctx.last_kernel == name
    sh = (n, nx * ny)
    return (ri.cpu().numpy().view(np.uint32).reshape(sh), x16.cpu().numpy().reshape(sh), dist.cpu().numpy().reshape(sh),
            du.cpu().numpy().view(np.uint16).reshape(sh), name)


def _check_vs_oracle(sub, left, right, p, ri, x16, dist):
    ex16, edist = sub.refine_subpixel(left, right, p, ri)
    bad = np.nonzero(x16 != ex16)
    assert len(bad[0]) == 0, "%d mismatches, first at %s: got %s expected %s" % (len(bad[0]), bad[1][:3], x16[bad][:3], ex16[bad][:3])
    if p.distance_kind == _abi.DIST_PINHOLE:
        assert dist.tobytes() == edist.tobytes()
    else:
        assert np.array_equal(dist == 0, edist == 0) and np.allclose(dist, edist, rtol=1e-12, atol=0, equal_nan=True)


# (channels, template, stride, cost, corr kernel option, expected sweep kernel)
FAMILIES = [
    (1, (16, 16), (1, 1), "sad", "auto", "dense_sad_argmin_kernel"),
    (3, (16, 16), (1, 1), "sad", "auto", "dense_sad_argmin_kernel"),
    (1, (16, 16), (1, 1), "ncc", "mma", "dense_corr_mma_kernel"),
    (1, (16, 16), (1, 1), "zncc", "mma", "dense_corr_mma_kernel"),
    (1, (16, 16), (1, 1), "ssd", "mma", "dense_corr_mma_kernel"),
    (3, (16, 16), (1, 1), "ncc", "mma", "dense_corr_mma_kernel"),
    (3, (16, 16), (1, 1), "zncc", "mma", "dense_corr_mma_kernel"),
    (3, (16, 16), (1, 1), "ssd", "mma", "dense_corr_mma_kernel"),
    (1, (16, 16), (1, 1), "ncc", "tcgen05", "dense_corr_umma_kernel"),
    (1, (16, 16), (1, 1), "zncc", "tcgen05", "dense_corr_umma_kernel"),
    (1, (15, 13), (2, 3), "sad", "auto", "block_cost_argmin_direct"),
    (3, (9, 7), (3, 2), "zncc", "auto", "block_cost_argmin_direct"),
    (2, (11, 5), (2, 1), "ssd", "auto", "block_cost_argmin_direct"),
    (4, (7, 6), (2, 2), "ncc", "auto", "block_cost_argmin_direct"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("side", [_abi.LEFT_CAM, _abi.RIGHT_CAM])
@pytest.mark.parametrize("fam", FAMILIES, ids=lambda f: "%s-c%d-%s" % (f[3], f[0], f[5]))
def test_device_equals_oracle_behind_every_sweep(ctx, sub, fam, side):
    c, (tw, th), (sx, sy), cost, kernel, expect = fam
    left, right = synth.make_pairs(2, 160, 40, c, shift=11 if side == _abi.LEFT_CAM else -11, noise_sigma=2.0, seed=c + tw)
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    for dist_kind in (_abi.DIST_PINHOLE, _abi.DIST_POWERLAW):
        # the direct form also takes a signed range (candidates on both sides of the window)
        p = _abi.make_params(tmpl_w=tw, tmpl_h=th, stride_x=sx, stride_y=sy, cost=cost, camera_side=side,
                             search_min=-4 if expect == "block_cost_argmin_direct" else 0, search_max=40, distance_kind=dist_kind)
        ri, x16, dist, _, name = _sweep_and_refine(ctx, left, right, p, kernel)
        assert name == expect
        assert (ri != _abi.NO_MATCH).any()
        _check_vs_oracle(sub, left, right, p, ri, x16, dist)


@pytest.mark.gpu
def test_c2_full_size(ctx, sub):
    """C2 geometry: 640x480 gray, 16x16 SAD, full range, every window; plus the invariants at size."""
    left, right = synth.make_pairs(2, 640, 480, 1, shift=37, noise_sigma=2.0, seed=325)
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad")
    ri, x16, dist, du, name = _sweep_and_refine(ctx, left, right, p)
    assert name == "dense_sad_argmin_kernel"
    _check_vs_oracle(sub, left, right, p, ri, x16, dist)
    both = (x16 != _abi.NO_SUBPIXEL) & (du != _abi.NO_DISPARITY)
    assert both.sum() > 0.5 * x16.size
    assert (np.abs(x16[both].astype(np.int64) - 16 * du[both].astype(np.int64)) <= 8).all()
    assert np.array_equal(x16 == _abi.NO_SUBPIXEL, ri == _abi.NO_MATCH)


@pytest.mark.gpu
def test_c3_sampled_rows(ctx, sub):
    """C3 geometry: 1280x720 colour, 32x32 ZNCC, D = 256; the oracle checks 24 window rows."""
    left, right = synth.make_pairs(1, 1280, 720, 3, shift=37, noise_sigma=2.0, seed=3)
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    p = _abi.make_params(tmpl_w=32, tmpl_h=32, cost="zncc", search_max=255)
    ri, x16, dist, du, name = _sweep_and_refine(ctx, left, right, p)
    f = _abi.frame_desc_for(left)
    nx, ny, _ = api.grid_dims(f, p)
    rows = np.random.default_rng(3).choice(ny, 24, replace=False)
    keep = np.zeros((1, ny, nx), bool)
    keep[:, rows] = True
    keep = keep.reshape(1, -1)
    ex16, edist = sub.refine_subpixel(left, right, p, np.where(keep, ri, _abi.NO_MATCH).astype(np.uint32))
    assert (ex16[keep] != _abi.NO_SUBPIXEL).any()
    assert np.array_equal(x16[keep], ex16[keep]) and dist[keep].tobytes() == edist[keep].tobytes()
    both = (x16 != _abi.NO_SUBPIXEL) & (du != _abi.NO_DISPARITY)
    assert (np.abs(x16[both].astype(np.int64) - 16 * du[both].astype(np.int64)) <= 8).all()
    assert np.array_equal(x16 == _abi.NO_SUBPIXEL, ri == _abi.NO_MATCH)


MASKS = [api.ALL_OUTPUTS, api.ALL_OUTPUTS | _abi.OUT_RESOLVED_DISPARITY_U16, _abi.OUT_RIGHT_INDEX,
         _abi.OUT_DISPARITY_U16 | _abi.OUT_RESOLVED_DISPARITY_U16, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("cost,c", [("sad", 1), ("zncc", 3), ("ssd", 1)])
def test_host_call_equals_match_dense(ctx, sub, cost, c):
    left, right = synth.make_pairs(2, 200, 48, c, shift=13, noise_sigma=2.0, seed=9)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost=cost, search_max=63)
    ri = ctx.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX)["right_index"]
    ex16, edist = sub.refine_subpixel(left, right, p, ri)
    for mask in MASKS:
        exp = ctx.match_dense(left, right, p, mask=mask)
        kernel = ctx.last_kernel
        got = ctx.match_dense_subpixel(left, right, p, mask=mask)
        assert ctx.last_kernel == kernel
        assert set(got) == set(exp) | {"disparity_x16", "subpixel_distance"}
        for k in exp:
            assert got[k].tobytes() == exp[k].tobytes(), (mask, k)
        assert np.array_equal(got["disparity_x16"], ex16) and got["subpixel_distance"].tobytes() == edist.tobytes()


@pytest.mark.gpu
def test_guard_against_non_candidates(ctx, sub):
    left, right = synth.make_pairs(1, 160, 40, 1, shift=11, noise_sigma=2.0, seed=21)
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_min=4, search_max=30)
    ri0, x160, _, _, _ = _sweep_and_refine(ctx, left, right, p)
    f = _abi.frame_desc_for(left)
    nx, ny, _ = api.grid_dims(f, p)
    nxc, nyc = f.width - p.tmpl_w + 1, f.height - p.tmpl_h + 1
    ri = ri0.copy()
    bad = {}
    w = 5 * nx + 80  # another row's index
    bad[w] = ri0[0, w] + nxc
    w = 6 * nx + 80  # x' in the frame, outside the search range (disparity 2 < search_min)
    bad[w] = 6 * nxc + 78
    w = 7 * nx + 80  # past the last position of the frame
    bad[w] = nxc * nyc + 3
    w = 8 * nx + 80
    bad[w] = 0xFFFFFFFE
    for k, v in bad.items():
        ri[0, k] = v
    _, x16, dist, _, _ = _sweep_and_refine(ctx, left, right, p, ri_override=ri)
    idx = np.array(sorted(bad))
    assert (x16[0, idx] == _abi.NO_SUBPIXEL).all() and (dist[0, idx] == 0.0).all()
    others = np.ones(x16.shape[1], bool)
    others[idx] = False
    assert np.array_equal(x16[0, others], x160[0, others])
    _check_vs_oracle(sub, left, right, p, ri, x16, dist)


@pytest.mark.gpu
@pytest.mark.parametrize("cost,c", [("sad", 1), ("zncc", 3), ("ssd", 4)])
def test_dirty_padding(ctx, cost, c):
    # widths whose rows end just past a word boundary, so the last words hold padding bytes
    left, right = synth.make_pairs(2, 157, 40, c, shift=9, noise_sigma=2.0, seed=c)
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    p = _abi.make_params(tmpl_w=13, tmpl_h=9, cost=cost, search_max=40)
    clean = _sweep_and_refine(ctx, left, right, p)
    for fill in (0xFF, "random"):
        dirty = _sweep_and_refine(ctx, left, right, p, fill=fill, seed=7)
        for a, b in zip(clean[:4], dirty[:4]):
            assert a.tobytes() == b.tobytes(), fill


@pytest.mark.gpu
def test_refusals(ctx):
    torch = pytest.importorskip("torch")
    left, right = synth.make_pairs(1, 64, 32, 1, shift=5, seed=1)
    dl, f = _device_frames(torch, left)
    p = _abi.make_params(tmpl_w=8, tmpl_h=8)
    ri = torch.zeros(4096, dtype=torch.int32, device="cuda")
    x16 = torch.zeros(4096, dtype=torch.int32, device="cuda")
    L = api.lib()

    def call(l, r, o_x16, o_dist):
        return L.usv_refine_subpixel_device(ctx._h, C.c_void_p(l), C.c_void_p(r), C.byref(f), C.c_int32(1), C.byref(p),
                                            C.c_void_p(ri.data_ptr()), C.c_void_p(o_x16), C.c_void_p(o_dist), C.c_void_p(0))
    base = dl.data_ptr()
    assert call(base, base, None, None) == _abi.USV_ERR_INVALID_ARG
    assert call(base + 1, base, x16.data_ptr(), None) == _abi.USV_ERR_INVALID_ARG
    assert call(base, base, x16.data_ptr(), None) == _abi.USV_OK
    h = np.ascontiguousarray(left)
    fh = _abi.frame_desc_for(h)
    assert L.usv_match_dense_subpixel_host(ctx._h, C.c_void_p(h.ctypes.data), C.c_void_p(h.ctypes.data), C.byref(fh), C.c_int32(1),
                                           C.byref(p), None, None, None) == _abi.USV_ERR_INVALID_ARG
    torch.cuda.synchronize()
