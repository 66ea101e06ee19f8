"""USV_COST_CENSUS: 3x3 census bytes compared by Hamming distance (include/usv_b200.h).

The oracle is tests/census_oracle.c, compiled into a temporary directory: direct form, with every census byte computed
on the fly from the frame. The library instead transforms whole frames first (usv_census.cu) and sweeps them with the
Hamming arm of the SAD sweep or the direct form, so the two share no code. On the CPU the oracle is checked against a
numpy restatement; on the GPU every output array must equal the oracle's byte for byte (distances to 1e-12 relative:
device pow against libm pow)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth

HERE = os.path.dirname(os.path.abspath(__file__))
DIST_RTOL = 1e-12
NEIGHBOURS = [(-1, -1), (0, -1), (1, -1), (-1, 0), (1, 0), (-1, 1), (0, 1), (1, 1)]  # (dx, dy), bit k = entry k
POPCOUNT = np.array([bin(i).count("1") for i in range(256)], np.uint32)
CENSUS_OUT = (_abi.OUT_MATCHES | _abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST | _abi.OUT_SCORE | _abi.OUT_DISTANCE | _abi.OUT_DISTANCE_F32
              | _abi.OUT_DISPARITY_U16)


# ---- the oracle -------------------------------------------------------------------------------------------------------
class CensusOracle:
    def __init__(self, so_path):
        self.L = C.CDLL(so_path)

    def match_dense(self, left, right, p, mask=CENSUS_OUT):
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        f = _abi.frame_desc_for(left)
        nx, ny, _ = api.grid_dims(f, p)
        n = left.shape[0]
        arrs, st = api._alloc_host_outputs(n * nx * ny, mask)
        rc = self.L.usv_census_oracle_match_dense(api._ptr(left), api._ptr(right), C.byref(f), C.c_int32(n), C.byref(p), C.byref(st))
        assert rc == 0
        return {k: v.reshape(n, nx * ny) for k, v in arrs.items()}

    def match_templates(self, left, right, tx, ty, p, mask=CENSUS_OUT, rows=False):
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        f = _abi.frame_desc_for(left)
        n, nt = left.shape[0], len(tx)
        tx, ty = np.ascontiguousarray(tx, np.int32), np.ascontiguousarray(ty, np.int32)
        arrs, st = api._alloc_host_outputs(n * nt, mask)
        cap = f.width
        cost_rows = np.full((n, nt, cap), 0xFFFFFFFF, np.uint32) if rows else None
        rc = self.L.usv_census_oracle_match_templates(api._ptr(left), api._ptr(right), C.byref(f), C.c_int32(n), api._ptr(tx), api._ptr(ty),
                                                      C.c_int32(nt), C.byref(p), C.byref(st), api._ptr(cost_rows), C.c_int32(cap))
        assert rc == 0
        out = {k: v.reshape(n, nt) for k, v in arrs.items()}
        if rows:
            out["cost_rows"] = cost_rows
        return out


@pytest.fixture(scope="module")
def census_oracle(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("census_oracle") / "libusv_census_oracle.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"  # as oracle/Makefile: the system compiler has OpenMP
    out = subprocess.run([cc, "-O3", "-fopenmp", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "census_oracle.c"), "-lm"],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return CensusOracle(so)


# ---- numpy restatement ------------------------------------------------------------------------------------------------
def census_np(frame):
    """[H, W] or [H, W, C] uint8 -> census bytes: shifted comparisons, neighbours outside the frame never darker."""
    f = frame.astype(np.int16)
    h, w = f.shape[:2]
    pad = np.full((h + 2, w + 2) + f.shape[2:], 256, np.int16)
    pad[1:-1, 1:-1] = f
    out = np.zeros(f.shape, np.uint8)
    for k, (dx, dy) in enumerate(NEIGHBOURS):
        out |= (pad[1 + dy:1 + dy + h, 1 + dx:1 + dx + w] < f).astype(np.uint8) << k
    return out


def restated_window(ctl, ctr, x, y, p, nxc):
    """(candidates x' ascending, their Hamming costs) of the window at (x, y)."""
    d = np.arange(p.search_min, min(p.search_max, 4 * nxc) + 1)
    xr = x - d if p.camera_side == _abi.LEFT_CAM else x + d
    xr = np.unique(xr[(xr >= 0) & (xr < nxc)])
    a = ctl[y:y + p.tmpl_h, x:x + p.tmpl_w]
    costs = np.array([POPCOUNT[a ^ ctr[y:y + p.tmpl_h, c:c + p.tmpl_w]].sum() for c in xr], np.uint32)
    return xr, costs


def restated_winner(ctl, ctr, x, y, p, nxc, n):
    """(right_index, raw_cost, disparity_u16, MatchValue) by brute force: np.argmin is the first minimum."""
    xr, costs = restated_window(ctl, ctr, x, y, p, nxc)
    if len(xr) == 0:
        return _abi.NO_MATCH, 0xFFFFFFFF, _abi.NO_DISPARITY, np.inf
    j = int(np.argmin(costs))
    v = float(costs[j]) / float(8 * n)
    ok = v < p.accept_threshold
    d = x - xr[j] if p.camera_side == _abi.LEFT_CAM else xr[j] - x
    return (y * nxc + int(xr[j]) if ok else _abi.NO_MATCH), int(costs[j]), (int(d) & 0xFFFF if ok else _abi.NO_DISPARITY), v


def _frames(n, h, w, c, seed, shift=5):
    left, right = synth.make_pairs(n, w, h, c, shift=shift, noise_sigma=3.0, seed=seed)
    left[:, : h // 4, : w // 3] = 128  # a flat patch: ties between candidates
    return left, right


CPU_CASES = [  # (w, h, c, tw, th, kw)
    (40, 14, 1, 5, 4, dict()),
    (37, 12, 1, 4, 3, dict(camera_side=_abi.RIGHT_CAM, search_max=12)),
    (30, 11, 3, 3, 3, dict(search_min=-6, search_max=9, accept_threshold=0.3)),
    (33, 13, 3, 6, 2, dict(camera_side=_abi.RIGHT_CAM, search_min=-4, search_max=20)),
    (41, 15, 1, 7, 5, dict(stride_x=2, stride_y=3, search_max=15)),
    (26, 10, 2, 4, 4, dict(search_min=2, search_max=14)),
]


@pytest.mark.parametrize("w,h,c,tw,th,kw", CPU_CASES)
def test_oracle_matches_numpy_restatement(census_oracle, w, h, c, tw, th, kw):
    left, right = _frames(2, h, w, c, seed=w * h + c)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="census", **kw)
    got = census_oracle.match_dense(left, right, p)
    nxc, nyc = w - tw + 1, h - th + 1
    n = tw * th * c
    for pr in range(2):
        ctl, ctr = census_np(left[pr]), census_np(right[pr])
        k = 0
        for y in range(0, nyc, p.stride_y):
            for x in range(0, nxc, p.stride_x):
                ri, raw, disp, v = restated_winner(ctl, ctr, x, y, p, nxc, n)
                assert got["right_index"][pr, k] == ri and got["raw_cost"][pr, k] == raw, (pr, x, y)
                assert got["disparity_u16"][pr, k] == disp and got["matches"]["LeftIndex"][pr, k] == k
                assert got["matches"]["MatchValue"][pr, k] == v and got["score"][pr, k] == 0.0
                k += 1
        assert k == got["right_index"].shape[1]


@pytest.mark.parametrize("c,side", [(1, _abi.LEFT_CAM), (3, _abi.RIGHT_CAM)])
def test_oracle_sparse_cost_rows_match_numpy_restatement(census_oracle, c, side):
    w, h, tw, th = 36, 12, 5, 3
    left, right = _frames(1, h, w, c, seed=11 + c)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="census", camera_side=side, search_min=-3, search_max=17)
    rng = np.random.default_rng(c)
    tx = rng.integers(0, w - tw + 1, 25)
    ty = rng.integers(0, h - th + 1, 25)
    got = census_oracle.match_templates(left, right, tx, ty, p, rows=True)
    ctl, ctr = census_np(left[0]), census_np(right[0])
    for i, (x, y) in enumerate(zip(tx, ty)):
        xr, costs = restated_window(ctl, ctr, int(x), int(y), p, w - tw + 1)
        row = got["cost_rows"][0, i]
        assert np.array_equal(row[: len(costs)], costs) and (row[len(costs):] == 0xFFFFFFFF).all()
        ri, raw, disp, v = restated_winner(ctl, ctr, int(x), int(y), p, w - tw + 1, tw * th * c)
        assert (got["right_index"][0, i], got["raw_cost"][0, i], got["disparity_u16"][0, i]) == (ri, raw, disp)


def _increasing_lut(rng):
    """A random map of 0..127 into 0..255, strictly increasing (on uint8 only the identity is strictly increasing on all
    256 values, so the frames it maps hold values below 128)."""
    lut = np.full(256, 255, np.uint8)
    lut[:128] = np.sort(rng.choice(256, 128, replace=False))
    return lut


def test_strictly_increasing_lut_changes_nothing_in_the_oracle(census_oracle):
    rng = np.random.default_rng(7)
    lut = _increasing_lut(rng)
    assert (np.diff(lut[:128].astype(int)) > 0).all() and not np.array_equal(lut[:128], np.arange(128))
    for c in (1, 3):
        left, right = _frames(2, 16, 44, c, seed=5 + c)
        left, right = left >> 1, right >> 1
        p = _abi.make_params(tmpl_w=6, tmpl_h=5, cost="census", search_max=20)
        base = census_oracle.match_dense(left, right, p)
        for l2, r2 in ((lut[left], right), (left, lut[right]), (lut[left], lut[right])):
            got = census_oracle.match_dense(l2, r2, p)
            for k, v in base.items():
                assert got[k].tobytes() == v.tobytes(), k


def test_census_is_robust_to_a_brightness_map_where_sad_is_not(census_oracle, oracle):
    """A known shift, and the right camera through gamma 0.6 and gain 1.3 (clipped): on textured windows census finds the
    true disparity on nearly all of them, SAD on few. Measured on these inputs (3136 windows): census 1.00, SAD 0.18;
    the bounds leave room for a different libm or compiler without letting the two come close."""
    shift, w, h, tw = 12, 120, 40, 9
    left, right = synth.make_pairs(1, w, h, 1, shift=shift, noise_sigma=2.0, seed=21)
    lut = np.clip(np.round(255.0 * 1.3 * (np.arange(256) / 255.0) ** 0.6), 0, 255).astype(np.uint8)
    right = np.ascontiguousarray(lut[right])
    left = np.ascontiguousarray(left)
    kw = dict(tmpl_w=tw, tmpl_h=tw, search_max=40, accept_threshold=2.0)
    got_c = census_oracle.match_dense(left, right, _abi.make_params(cost="census", **kw), mask=_abi.OUT_DISPARITY_U16)
    got_s = oracle.match_dense(left, right, _abi.make_params(cost="sad", **kw), mask=_abi.OUT_DISPARITY_U16)
    nxc, nyc = w - tw + 1, h - tw + 1
    win = np.lib.stride_tricks.sliding_window_view(left[0].astype(np.float64), (tw, tw))[:nyc, :nxc]
    textured = win.std(axis=(2, 3)) > 20.0
    textured[:, : shift + 2] = False  # windows whose true match lies outside the right frame
    dc = got_c["disparity_u16"][0].reshape(nyc, nxc)
    ds = got_s["disparity_u16"][0].reshape(nyc, nxc)
    frac_c, frac_s = (dc[textured] == shift).mean(), (ds[textured] == shift).mean()
    assert textured.sum() > 500
    assert frac_c >= 0.9 and frac_s <= 0.5 and frac_c > frac_s + 0.4, (frac_c, frac_s)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _resolved_expected(oracle, winners, disparity):
    alive = np.zeros(len(winners), bool)
    kept = oracle.resolve_match_list(winners[winners["RightIndex"] != _abi.NO_MATCH])
    alive[np.unique(kept["LeftIndex"])] = True
    return np.where(alive, disparity, _abi.NO_DISPARITY).astype(np.uint16)


def _compare(got, exp):
    for k in ("right_index", "raw_cost", "raw_cost_u16", "disparity_u16", "resolved_disparity_u16", "score"):
        if k in got and k in exp:
            assert got[k].tobytes() == exp[k].tobytes(), k
    if "matches" in got:
        assert got["matches"].tobytes() == exp["matches"].tobytes()
    for k, tol in (("distance", DIST_RTOL), ("distance_f32", 1e-6)):
        if k in got:
            g, e = got[k].astype(np.float64), exp[k].astype(np.float64)
            assert np.array_equal(np.isinf(g), np.isinf(e)) and np.array_equal(g == 0, e == 0), k
            fin = np.isfinite(e)
            assert np.allclose(g[fin], e[fin], rtol=tol, atol=0), k


def _expected(census_oracle, oracle, left, right, p, resolved):
    exp = census_oracle.match_dense(left, right, p)
    if 8 * p.tmpl_w * p.tmpl_h * (left[0, 0, 0].size) < 0xFFFF:
        exp["raw_cost_u16"] = exp["raw_cost"].astype(np.uint16)
    if resolved:
        exp["resolved_disparity_u16"] = np.stack([_resolved_expected(oracle, exp["matches"][i], exp["disparity_u16"][i])
                                                  for i in range(len(left))])
    return exp


def _mask(p, c, resolved):
    m = api.ALL_OUTPUTS
    if 8 * p.tmpl_w * p.tmpl_h * c < 0xFFFF:
        m |= _abi.OUT_RAW_COST_U16
    return m | (_abi.OUT_RESOLVED_DISPARITY_U16 if resolved else 0)


L_, R_ = _abi.LEFT_CAM, _abi.RIGHT_CAM
SWEEP_CASES = [  # (w, h, c, tw, th, side, kw): every variant of dense_census_argmin_kernel
    (120, 24, 1, 16, 16, L_, dict(search_max=30)),                       # gray JT = 4, one ring
    (160, 24, 1, 16, 16, R_, dict(search_max=100)),                      # gray JT = 8
    (150, 30, 1, 16, 16, L_, dict(search_min=3)),                        # full range, thin pass / fold
    (100, 20, 1, 8, 1, L_, dict(search_max=40)),                         # th = 1
    (110, 40, 1, 12, 17, R_, dict(search_min=-10, search_max=30)),       # two-half ring, negative range
    (90, 70, 1, 24, 64, L_, dict(search_max=60)),                        # th = 64, JT = 8
    (100, 30, 1, 32, 8, R_, dict(search_min=-20, search_max=20)),        # tw = 32
    (96, 22, 3, 8, 8, L_, dict(search_max=60)),                          # colour JT = 8
    (80, 22, 3, 16, 4, R_, dict(search_min=-8, search_max=20, accept_threshold=0.25)),  # colour JT = 4
    (72, 70, 3, 12, 64, L_, dict(search_max=30)),                        # colour th = 64
    (64, 40, 3, 24, 17, R_, dict(search_max=50)),                        # colour tw = 24, th = 17
    (70, 26, 1, 12, 16, L_, dict(search_min=-15, search_max=-2)),        # an all-negative range
]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,c,tw,th,side,kw", SWEEP_CASES)
def test_census_sweep_equals_oracle(ctx, census_oracle, oracle, w, h, c, tw, th, side, kw):
    left, right = _frames(2, h, w, c, seed=w + 7 * h + c, shift=7 if side == L_ else -7)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="census", camera_side=side, **kw)
    got = ctx.match_dense(left, right, p, mask=_mask(p, c, True))
    assert ctx.last_kernel == "dense_census_argmin_kernel"
    _compare(got, _expected(census_oracle, oracle, left, right, p, True))


DIRECT_CASES = [  # (w, h, c, tw, th, side, kw): what the sweep does not cover
    (80, 24, 1, 20, 8, L_, dict(search_max=40)),                         # tw = 20
    (60, 72, 1, 8, 65, R_, dict(search_max=30)),                         # th = 65
    (50, 20, 2, 6, 6, L_, dict(search_min=-4, search_max=20)),           # C = 2
    (50, 20, 4, 5, 5, R_, dict(search_max=15, accept_threshold=0.3)),    # C = 4
    (90, 30, 1, 16, 16, L_, dict(stride_x=2, search_max=40)),            # stride 2
    (60, 26, 3, 9, 7, R_, dict(stride_x=2, stride_y=3, search_max=25)),  # colour, odd width, strides
]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,c,tw,th,side,kw", DIRECT_CASES)
def test_census_direct_form_equals_oracle(ctx, census_oracle, oracle, w, h, c, tw, th, side, kw):
    left, right = _frames(2, h, w, c, seed=w + 5 * h + c, shift=6 if side == L_ else -6)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="census", camera_side=side, **kw)
    dense = p.stride_x == 1 and p.stride_y == 1
    got = ctx.match_dense(left, right, p, mask=_mask(p, c, dense))
    assert ctx.last_kernel == "block_cost_argmin_direct"
    _compare(got, _expected(census_oracle, oracle, left, right, p, dense))


@pytest.mark.gpu
@pytest.mark.parametrize("c,side", [(1, L_), (3, R_), (2, L_)])
def test_census_sparse_templates_equal_oracle(ctx, census_oracle, c, side):
    w, h, tw, th = 90, 30, 12, 10
    left, right = _frames(2, h, w, c, seed=3 * c)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="census", camera_side=side, search_min=-5, search_max=40)
    rng = np.random.default_rng(c)
    tx, ty = rng.integers(0, w - tw + 1, 60), rng.integers(0, h - th + 1, 60)
    got = ctx.match_templates(left, right, tx, ty, p, mask=api.ALL_OUTPUTS | _abi.OUT_RAW_COST_U16, rows=True)
    assert ctx.last_kernel == "block_cost_argmin_direct"
    exp = census_oracle.match_templates(left, right, tx, ty, p, rows=True)
    exp["raw_cost_u16"] = exp["raw_cost"].astype(np.uint16)
    _compare(got, exp)
    assert got["cost_rows"].tobytes() == exp["cost_rows"].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("geom", ["C2", "C3"])
def test_census_full_geometry_sampled_rows(ctx, census_oracle, geom):
    """One pair at the C2 (640x480 gray, 16x16, full range) and C3 (1280x720x3, 32x32, D = 256) geometries; whole window
    rows checked against the oracle (as a template list), the first, the last and one inside."""
    if geom == "C2":
        w, h, c, tw, kw = 640, 480, 1, 16, dict()
    else:
        w, h, c, tw, kw = 1280, 720, 3, 32, dict(search_max=255)
    left, right = synth.make_pairs(1, w, h, c, shift=37, noise_sigma=2.0, seed=9)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=tw, cost="census", **kw)
    got = ctx.match_dense(left, right, p)
    assert ctx.last_kernel == "dense_census_argmin_kernel"
    nxc, nyc = w - tw + 1, h - tw + 1
    for y in (0, nyc // 2 + 3, nyc - 1) if geom == "C2" else (nyc - 1,):
        tx = np.arange(nxc)
        exp = census_oracle.match_templates(left, right, tx, np.full(nxc, y), p)
        sl = slice(y * nxc, (y + 1) * nxc)
        row = {k: v[:, sl] for k, v in got.items()}
        exp["matches"]["LeftIndex"] += y * nxc
        _compare(row, exp)


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 3])
def test_census_device_invariant_to_increasing_lut(ctx, c):
    rng = np.random.default_rng(40 + c)
    lut = _increasing_lut(rng)
    left, right = _frames(2, 40, 150, c, seed=c)
    left, right = left >> 1, right >> 1
    for p in (_abi.make_params(tmpl_w=16, tmpl_h=16, cost="census", search_max=90),
              _abi.make_params(tmpl_w=10, tmpl_h=9, cost="census", search_max=50)):
        base = ctx.match_dense(left, right, p, mask=_mask(p, c, True))
        k0 = ctx.last_kernel
        for l2, r2 in ((left, lut[right]), (lut[left], right)):
            got = ctx.match_dense(np.ascontiguousarray(l2), np.ascontiguousarray(r2), p, mask=_mask(p, c, True))
            assert ctx.last_kernel == k0
            for k, v in base.items():
                assert got[k].tobytes() == v.tobytes(), k


def _dirty_device_run(ctx, left, right, p, mask, fill, rng):
    """match_dense_device on frames whose row padding and inter-frame gaps hold `fill` (a byte or "random")."""
    torch = pytest.importorskip("torch")
    n, h = left.shape[:2]
    rb = left[0, 0].size
    row_stride = ((rb + 15) & ~15) + 16
    frame_stride = h * row_stride + 48
    outs, st = {}, _abi.Outputs()
    devs = []
    for fr in (left, right):
        total = (n - 1) * frame_stride + h * row_stride
        buf = rng.integers(0, 256, total, dtype=np.uint8) if fill == "random" else np.full(total, fill, np.uint8)
        view = np.lib.stride_tricks.as_strided(buf, shape=fr.shape, strides=(frame_stride, row_stride) + fr.strides[2:])
        view[...] = fr
        devs.append(torch.from_numpy(buf).cuda())
    f = _abi.FrameDesc(left.shape[2], h, left[0, 0, 0].size, row_stride, frame_stride)
    nx, ny, _ = api.grid_dims(f, p)
    for name, bit, dt in _abi.OUTPUT_FIELDS:
        if mask & bit:
            outs[name] = torch.zeros(n * nx * ny * dt.itemsize, dtype=torch.uint8, device="cuda")
            setattr(st, name, outs[name].data_ptr())
    ctx.match_dense_device(devs[0].data_ptr(), devs[1].data_ptr(), f, n, p, st, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    dts = {name: dt for name, _, dt in _abi.OUTPUT_FIELDS}
    return {k: v.cpu().numpy().view(dts[k]).reshape(n, nx * ny) for k, v in outs.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("c,tw,kernel", [(1, 16, "dense_census_argmin_kernel"), (3, 8, "dense_census_argmin_kernel"),
                                         (1, 20, "block_cost_argmin_direct"), (3, 7, "block_cost_argmin_direct")])
@pytest.mark.parametrize("fill", [0xFF, "random"])
def test_census_dirty_row_padding_changes_nothing(ctx, c, tw, kernel, fill):
    left, right = _frames(2, 30, 101, c, seed=tw)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=8, cost="census", search_max=45)
    mask = _mask(p, c, True)
    exp = ctx.match_dense(left, right, p, mask=mask)
    got = _dirty_device_run(ctx, left, right, p, mask, fill, np.random.default_rng(3))
    assert ctx.last_kernel == kernel
    for k, v in exp.items():
        assert got[k].tobytes() == v.tobytes(), k


@pytest.mark.gpu
def test_census_split_batch_equals_unsplit_batches(ctx):
    """Colour census at 1280x720, 8x8: the pair scratch (capped at 1.5 GB, usv_capi.cu: kPairScratchCap) holds the census
    frames and colour planes of both cameras for some 145 pairs, so this batch runs in two chunks, the second partly
    filled. Each must give what the same pairs give in batches that fit one chunk."""
    w, h, c, tw = 1280, 720, 3, 8
    pitch = (w * c + 15) & ~15
    per_pair = 2 * pitch * h + 2 * c * h * (((w + 15) & ~15) + 16)
    cap_pairs = (3 << 29) // per_pair
    n = cap_pairs + cap_pairs // 4 + max(1, cap_pairs // 8) + 1
    small = max(1, cap_pairs // 2)
    assert cap_pairs < n < 2 * cap_pairs
    rng = np.random.default_rng(n)
    left = rng.integers(0, 256, size=(n, h, w, c), dtype=np.uint8)
    right = np.roll(left, -9, axis=2)
    right[:, ::7] ^= 0x11
    p = _abi.make_params(tmpl_w=tw, tmpl_h=tw, search_max=64, cost="census")
    for mask in (_abi.OUT_DISPARITY_U16, _abi.OUT_RAW_COST_U16):
        before = ctx.launch_count
        ctx.match_dense(left[:1], right[:1], p, mask=mask)
        per_chunk = ctx.launch_count - before
        before = ctx.launch_count
        got = ctx.match_dense(left, right, p, mask=mask)
        assert ctx.last_kernel == "dense_census_argmin_kernel"
        assert ctx.launch_count - before == 2 * per_chunk
        for p0 in range(0, n, small):
            exp = ctx.match_dense(left[p0:p0 + small], right[p0:p0 + small], p, mask=mask)
            for name, arr in exp.items():
                assert got[name][p0:p0 + small].tobytes() == arr.tobytes(), (name, p0)
        del got


@pytest.mark.gpu
def test_census_stream_submit_equals_match_dense(ctx):
    left, right = _frames(4, 40, 160, 1, seed=12, shift=11)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="census", search_max=63)
    f = _abi.frame_desc_for(left)
    mask = _abi.OUT_RESOLVED_DISPARITY_U16 | _abi.OUT_RAW_COST_U16 | _abi.OUT_RIGHT_INDEX
    exp = ctx.match_dense(left, right, p, mask=mask)
    st = ctx.stream(f, p, pairs_per_slot=2, n_slots=2, mask=mask)
    try:
        for s in range(2):
            st.slots[s]["left"][...] = left[2 * s:2 * s + 2]
            st.slots[s]["right"][...] = right[2 * s:2 * s + 2]
            st.submit(s)
        for s in range(2):
            st.wait(s)
            for k, v in st.slots[s]["out"].items():
                assert v.tobytes() == exp[k][2 * s:2 * s + 2].tobytes(), (s, k)
    finally:
        st.close()
    assert ctx.last_kernel == "dense_census_argmin_kernel"


@pytest.mark.gpu
def test_census_block_search_host_is_generate_resolve_distance(ctx, census_oracle, oracle):
    """usv_block_search_host with census = the oracle's winners through ResolveMatchList (oracle/block_search_oracle.c's
    restatement, checked against the reference's own lines by test_oracle_vs_ref.py), with each entry's distance."""
    left, right = synth.make_pairs(1, 150, 36, 1, shift=9, noise_sigma=2.0, seed=5)
    left[0, :, 100:] = 60
    p = _abi.make_params(tmpl_w=12, tmpl_h=12, cost="census", search_max=60, distance_kind=_abi.DIST_POWERLAW)
    got_m, got_d = ctx.block_search(left[0], right[0], p)
    assert ctx.last_kernel == "dense_census_argmin_kernel"
    exp = census_oracle.match_dense(left, right, p)
    win = exp["matches"][0]
    kept = win[win["RightIndex"] != _abi.NO_MATCH]
    exp_list = oracle.resolve_match_list(kept)
    assert len(exp_list) > 0 and got_m.tobytes() == exp_list.tobytes()
    exp_d = exp["distance"][0][exp_list["LeftIndex"]]
    assert np.array_equal(np.isinf(got_d), np.isinf(exp_d))
    fin = np.isfinite(exp_d)
    assert np.allclose(got_d[fin], exp_d[fin], rtol=DIST_RTOL, atol=0)


@pytest.mark.gpu
def test_census_refusals_and_kernel_choice(ctx):
    left, right = _frames(1, 30, 90, 3, seed=1)
    p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="census", search_max=40)
    with pytest.raises(api.UsvError, match=r"\(-4\)"):
        ctx.match_dense_subpixel(left, right, p)
    torch = pytest.importorskip("torch")
    f = _abi.FrameDesc(64, 16, 1, 64, 64 * 16)
    d = torch.zeros(64 * 16, dtype=torch.uint8, device="cuda")
    ri = torch.zeros(57 * 9, dtype=torch.int32, device="cuda")
    q = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="census", search_max=40)
    with pytest.raises(api.UsvError, match=r"\(-4\)"):
        ctx.refine_subpixel_device(d.data_ptr(), d.data_ptr(), f, 1, q, ri.data_ptr(), ri.data_ptr())
    # raw_cost_u16: 8 n < 0xFFFF is served (32x64x3: n = 6144), 8 n >= 0xFFFF refused (32x256: n = 8192)
    big = _abi.make_params(tmpl_w=32, tmpl_h=64, cost="census", search_max=8)
    lf, rt = _frames(1, 66, 40, 3, seed=2)
    ctx.match_dense(lf, rt, big, mask=_abi.OUT_RAW_COST_U16)
    tall = _abi.make_params(tmpl_w=32, tmpl_h=256, cost="census", search_max=8)
    lf, rt = _frames(1, 258, 40, 1, seed=2)
    with pytest.raises(api.UsvError, match=r"\(-4\)"):
        ctx.match_dense(lf, rt, tall, mask=_abi.OUT_RAW_COST_U16)
    # no correlation sweep takes census, whichever one is forced
    for which in ("alu", "mma", "tcgen05"):
        ctx.corr_kernel(which)
        try:
            ctx.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX)
            assert ctx.last_kernel == "dense_census_argmin_kernel", which
        finally:
            ctx.corr_kernel("auto")
