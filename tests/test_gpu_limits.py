"""The matching kernels at the edges the synthetic frames of the other suites never reach.

  * Saturated inputs at every integer limit the kernels rely on: the SAD key `cost << xb | code` below bit 31
    (usv_dense.cu), s32 Sab in the mma.sync and tcgen05 kernels, u32 SSD scoring below 2^28 in mma.sync, the tcgen05 band
    height that keeps its running row sums below 2^31, raw_cost_u16 below its "no candidate" value, the 2048-window rows
    of the resolved map, the row-chunked strips and the shared-memory envelope of the direct form. Each case sits just
    inside or just outside a limit and names the kernel that served it (usv_last_kernel).
  * Dirty row padding: every kernel family on frames whose stride padding (and inter-frame gap) holds 0xFF or random
    bytes, reached through the device entry points, the stream ring (which copies the caller's padding verbatim when its
    pitch matches) and the host path (whose grow-only staging keeps the bytes of an earlier call).

The reference is an independent int64 numpy restatement (`reference_dense`): box sums of |a-b|, a*b and the window
statistics by cumulative sums, scored with the same correctly rounded f64 operations as the device, first minimum in
ascending x'. The CPU tests at the top pin it to the C oracle, including the largest template (32768 bytes) on
saturated frames; the C oracle is too slow for 32x1024 templates over whole frames."""
import ctypes as C

import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth

INT_MASK = _abi.OUT_MATCHES | _abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST | _abi.OUT_DISPARITY_U16
FLOAT_MASK = _abi.OUT_MATCHES | _abi.OUT_RIGHT_INDEX | _abi.OUT_SCORE | _abi.OUT_DISPARITY_U16
ACCEPT_ALL = 3.0  # every MatchValue (SAD/SSD <= 1, NCC/ZNCC <= 2) is accepted: every winner is visible in right_index


# ---- the reference -------------------------------------------------------------------------------------------------
def _box(img, th, wb, c, nxc, nyc):
    """Sums of img [H, W*C] int64 over th rows x wb bytes of the window whose first byte is x*c, for every (y, x)."""
    h, w = img.shape
    ii = np.zeros((h + 1, w + 1), np.int64)
    ii[1:, 1:] = img.cumsum(0).cumsum(1)
    rows = ii[th:th + nyc] - ii[:nyc]
    xs = np.arange(nxc) * c
    return rows[:, xs + wb] - rows[:, xs]


def _shift_bytes(r, sb):
    """out[:, u] = r[:, u + sb] where that exists, else 0."""
    out = np.zeros_like(r)
    w = r.shape[1]
    if sb >= 0:
        out[:, :w - sb] = r[:, sb:]
    else:
        out[:, -sb:] = r[:, :w + sb]
    return out


def _scores(kind, n, sab, sa, sb, saa, sbb):
    """NCC / ZNCC from exact int64 sums with the device's operations (usv_common.cuh: ncc_score, zncc_score)."""
    if kind == _abi.COST_NCC:
        num, da, db = sab, saa, sbb
    else:
        num, da, db = n * sab - sa * sb, n * saa - sa * sa, n * sbb - sb * sb
    zero = (da == 0) | (db == 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        sc = num.astype(np.float64) * (1.0 / np.sqrt(da.astype(np.float64))) * (1.0 / np.sqrt(db.astype(np.float64)))
    return np.where(zero, 0.0, sc)


def reference_dense(left, right, p):
    """Dense stride-1 sweep of every pair in int64 numpy: dict of [n, nyc*nxc] arrays (matches, right_index, raw_cost,
    score, disparity_u16) as include/usv_b200.h defines them."""
    assert p.stride_x == 1 and p.stride_y == 1
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    n, h, w = left.shape[:3]
    c = left.shape[3] if left.ndim == 4 else 1
    tw, th, kind = p.tmpl_w, p.tmpl_h, p.cost_kind
    nxc, nyc = w - tw + 1, h - th + 1
    ne, wb = tw * th * c, tw * c
    integer = kind <= _abi.COST_SSD
    xs = np.arange(nxc)
    out = {"right_index": [], "raw_cost": [], "score": [], "disparity_u16": [], "matches": []}
    for i in range(n):
        L = left[i].reshape(h, w * c).astype(np.int64)
        R = right[i].reshape(h, w * c).astype(np.int64)
        box = lambda img: _box(img, th, wb, c, nxc, nyc)  # noqa: E731
        sa, saa, sb_all, sbb_all = box(L), box(L * L), box(R), box(R * R)
        best_raw = np.full((nyc, nxc), -1, np.int64)
        best_v = np.full((nyc, nxc), np.inf)
        best_sc = np.zeros((nyc, nxc))
        best_x = np.full((nyc, nxc), -1, np.int64)
        # x' = x + s; ascending x' = ascending s, so a strict '<' keeps the first minimum (P/Main.cpp:451)
        if p.camera_side == _abi.LEFT_CAM:
            s_lo, s_hi = -p.search_max, -p.search_min
        else:
            s_lo, s_hi = p.search_min, p.search_max
        for s in range(max(s_lo, -(nxc - 1)), min(s_hi, nxc - 1) + 1):
            xr = xs + s
            ok = (xr >= 0) & (xr <= nxc - 1)
            xrc = np.clip(xr, 0, nxc - 1)
            Rs = _shift_bytes(R, s * c)
            if kind == _abi.COST_SAD:
                cost = box(np.abs(L - Rs))
            else:
                sab = box(L * Rs)
                sb, sbb = sb_all[:, xrc], sbb_all[:, xrc]
                if kind == _abi.COST_SSD:
                    cost = saa + sbb - 2 * sab
                else:
                    sc = _scores(kind, ne, sab, sa, sb, saa, sbb)
                    v = 1.0 - sc
            if integer:
                better = ok[None, :] & ((best_raw < 0) | (cost < best_raw))
                best_raw = np.where(better, cost, best_raw)
            else:
                better = ok[None, :] & (v < best_v)
                best_v = np.where(better, v, best_v)
                best_sc = np.where(better, sc, best_sc)
            best_x = np.where(better, xr[None, :], best_x)
        has = best_x >= 0
        if integer:
            den = float(255 * ne) if kind == _abi.COST_SAD else float(65025 * ne)
            best_v = np.where(has, best_raw / den, np.inf)
            raw = np.where(has, best_raw, 0xFFFFFFFF).astype(np.uint32)
            score = np.zeros((nyc, nxc))
        else:
            raw = np.full((nyc, nxc), 0xFFFFFFFF, np.uint32)
            score = np.where(has, best_sc, 0.0)
        acc = has & (best_v < p.accept_threshold)
        y = np.arange(nyc)[:, None]
        d = (xs[None, :] - best_x) if p.camera_side == _abi.LEFT_CAM else (best_x - xs[None, :])
        ri = np.where(acc, y * nxc + best_x, _abi.NO_MATCH).astype(np.uint32)
        m = np.zeros(nyc * nxc, _abi.MATCH_DTYPE)
        m["LeftIndex"] = np.arange(nyc * nxc)
        m["RightIndex"] = ri.ravel()
        m["MatchValue"] = best_v.ravel()
        out["right_index"].append(ri.ravel())
        out["raw_cost"].append(raw.ravel())
        out["score"].append(score.ravel())
        out["disparity_u16"].append(np.where(acc, d & 0xFFFF, _abi.NO_DISPARITY).astype(np.uint16).ravel())
        out["matches"].append(m)
    return {k: np.stack(v) for k, v in out.items()}


def reference_candidates(left, right, x, y, p, pair=0):
    """Every candidate of the template at (x, y) in scan order: (x' array, integer costs or f64 scores)."""
    L, R = left[pair].astype(np.int64), right[pair].astype(np.int64)
    w = L.shape[1]
    tw, th = p.tmpl_w, p.tmpl_h
    nxc = w - tw + 1
    if p.camera_side == _abi.LEFT_CAM:
        lo, hi = x - p.search_max, x - p.search_min
    else:
        lo, hi = x + p.search_min, x + p.search_max
    xr = np.arange(max(lo, 0), min(hi, nxc - 1) + 1)
    t = L[y:y + th, x:x + tw].reshape(-1)
    cands = np.stack([R[y:y + th, j:j + tw].reshape(-1) for j in xr]) if len(xr) else np.zeros((0, t.size), np.int64)
    if p.cost_kind == _abi.COST_SAD:
        return xr, np.abs(cands - t).sum(1)
    if p.cost_kind == _abi.COST_SSD:
        return xr, ((cands - t) ** 2).sum(1)
    sab, sb, sbb = (cands * t).sum(1), cands.sum(1), (cands * cands).sum(1)
    ones = np.ones_like(sab)
    return xr, _scores(p.cost_kind, t.size, sab, ones * t.sum(), sb, ones * (t * t).sum(), sbb)


# ---- input patterns -------------------------------------------------------------------------------------------------
PATTERNS = ("saturated", "stripes", "dips")
PRODUCT_PATTERNS = PATTERNS + ("full",)  # "full": both frames 255, every product a*b is the maximum
SHIFT = 23  # the disparity the "dips" frames carry


def pattern(kind, n, h, w, c, camera_side=_abi.LEFT_CAM, seed=0):
    """saturated: left 255 / right 0, every candidate costs the maximum and the first one wins; stripes: 0/255 columns
    (periodic, so whole sets of candidates tie); dips: frames at 255 with a sparse sprinkle of random darker bytes, so
    sums sit near their maximum with nonzero variance, and the right frame carries a known shift."""
    shape = (n, h, w) if c == 1 else (n, h, w, c)
    if kind == "full":
        return np.full(shape, 255, np.uint8), np.full(shape, 255, np.uint8)
    if kind == "saturated":
        return np.full(shape, 255, np.uint8), np.zeros(shape, np.uint8)
    if kind == "stripes":
        col = np.where((np.arange(w + 3) // 3) % 2 == 0, 255, 0).astype(np.uint8)
        lf = np.broadcast_to(col[None, None, :w, None], (n, h, w, c))
        rt = np.broadcast_to(col[None, None, 1:w + 1, None], (n, h, w, c))
        return np.ascontiguousarray(lf.reshape(shape)), np.ascontiguousarray(rt.reshape(shape))
    rng = np.random.default_rng(seed)
    world = np.full((n, h, w + SHIFT, c), 255, np.uint8)
    dip = rng.random(world.shape) < 0.03
    world[dip] = rng.integers(0, 200, int(dip.sum()))
    a, b = world[:, :, :w], world[:, :, SHIFT:SHIFT + w]
    lf, rt = (a, b) if camera_side == _abi.LEFT_CAM else (b, a)
    return np.ascontiguousarray(lf.reshape(shape)), np.ascontiguousarray(rt.reshape(shape))


def _compare(got, exp, kind, what=""):
    integer = kind <= _abi.COST_SSD
    for k in ("right_index", "disparity_u16") + (("raw_cost",) if integer else ()):
        if k in got:
            bad = np.nonzero(got[k] != exp[k])
            assert len(bad[0]) == 0, "%s %s: %d mismatches, first at %s: got %s expected %s" % (
                what, k, len(bad[0]), bad[1][:1], got[k][bad][:3], exp[k][bad][:3])
    if not integer and "score" in got:
        assert got["score"].tobytes() == exp["score"].tobytes(), what + " score"
    if "matches" in got:
        gm, em = got["matches"], exp["matches"]
        assert np.array_equal(gm["RightIndex"], em["RightIndex"]) and np.array_equal(gm["LeftIndex"], em["LeftIndex"]), what
        assert gm["MatchValue"].tobytes() == em["MatchValue"].tobytes(), what + " MatchValue"


# ---- CPU: the reference against the C oracle ---------------------------------------------------------------------------
RANGES = {"full": dict(), "signed": dict(search_min=-9, search_max=9), "clipped": dict(search_min=3, search_max=20),
          "empty": dict(search_min=100, search_max=120)}


@pytest.mark.parametrize("rng_name", sorted(RANGES))
@pytest.mark.parametrize("side", [_abi.LEFT_CAM, _abi.RIGHT_CAM])
@pytest.mark.parametrize("cost", ["sad", "ssd", "ncc", "zncc"])
def test_reference_equals_oracle(oracle, cost, side, rng_name):
    for c, (tw, th) in ((1, (7, 5)), (3, (8, 4))):
        left, right = synth.make_pairs(2, 61, 19, c, shift=7, noise_sigma=2.0, seed=11 + c)
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        left[1, :9], right[1, :9] = 77, 77  # flat rows: every candidate ties, zero variance
        p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost=cost, camera_side=side, accept_threshold=0.4, **RANGES[rng_name])
        exp = oracle.match_dense(left, right, p, mask=_abi.OUT_MATCHES | _abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST |
                                 _abi.OUT_SCORE | _abi.OUT_DISPARITY_U16)
        got = reference_dense(left, right, p)
        for k in exp:
            assert got[k].tobytes() == exp[k].tobytes(), (c, k)


@pytest.mark.parametrize("pat", PATTERNS)
@pytest.mark.parametrize("cost", ["sad", "ssd", "ncc", "zncc"])
def test_reference_equals_oracle_at_the_largest_template(oracle, cost, pat):
    """32768-byte templates on saturated frames: the oracle's u32 SAD / SSD hold 65025 * 32768 = 2 130 739 200."""
    for c, tw, th in ((1, 32, 1024), (3, 32, 341)):
        left, right = pattern(pat, 1, th + 2, 40, c, seed=3)
        p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost=cost, search_min=-3, search_max=5, accept_threshold=ACCEPT_ALL)
        exp = oracle.match_dense(left, right, p, mask=_abi.OUT_MATCHES | _abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST |
                                 _abi.OUT_SCORE | _abi.OUT_DISPARITY_U16)
        got = reference_dense(left, right, p)
        for k in exp:
            assert got[k].tobytes() == exp[k].tobytes(), (c, k)
        if pat == "saturated" and cost in ("sad", "ssd"):
            assert (got["raw_cost"] == (255 if cost == "sad" else 65025) * tw * th * c).all()


def test_reference_candidates_equal_oracle_rows(oracle):
    left, right = pattern("dips", 1, 40, 90, 3, seed=8)
    for cost in ("sad", "zncc"):
        p = _abi.make_params(tmpl_w=9, tmpl_h=30, cost=cost, search_max=40)
        tx, ty = [0, 45, 81], [0, 5, 10]
        exp = oracle.match_templates(left, right, tx, ty, p, rows=True)
        for i, (x, y) in enumerate(zip(tx, ty)):
            xr, v = reference_candidates(left, right, x, y, p)
            rows = exp["cost_rows"] if cost == "sad" else exp["score_rows"]
            assert rows[0, i, :len(xr)].tobytes() == v.astype(rows.dtype).tobytes()


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _run_dense(ctx, left, right, p, mask, kernel="auto"):
    ctx.corr_kernel(kernel)
    try:
        return ctx.match_dense(left, right, p, mask=mask), ctx.last_kernel
    finally:
        ctx.corr_kernel("auto")


def _mask(cost):
    return INT_MASK if _abi.COST_NAMES[cost] <= _abi.COST_SSD else FLOAT_MASK


def _check_sampled(ctx, oracle, got, left, right, p, n_random, seed=0):
    """matches and distances of a dense result against the C oracle's answer for single windows: the frame's corners
    and edges plus n_random windows (pair 0). PINHOLE distances are IEEE divisions and products, so they are compared
    bit for bit; POWERLAW goes through the device's pow, which may differ from the host's in the last bit, so it is
    compared with the oracle to 1e-12 (as in test_gpu_parity.py) and bit for bit with the device's own distance table."""
    f = _abi.frame_desc_for(left)
    nxc, nyc = f.width - p.tmpl_w + 1, f.height - p.tmpl_h + 1
    rng = np.random.default_rng(seed)
    tx = np.r_[0, nxc - 1, 0, nxc - 1, nxc // 2, rng.integers(0, nxc, n_random)].astype(np.int32)
    ty = np.r_[0, 0, nyc - 1, nyc - 1, nyc // 2, rng.integers(0, nyc, n_random)].astype(np.int32)
    exp = oracle.match_templates(left[:1], right[:1], tx, ty, p, mask=_abi.OUT_MATCHES | _abi.OUT_DISTANCE)
    w_idx = ty.astype(np.int64) * nxc + tx
    gm, em = got["matches"][0][w_idx], exp["matches"][0]
    assert np.array_equal(gm["RightIndex"], em["RightIndex"]) and gm["MatchValue"].tobytes() == em["MatchValue"].tobytes()
    assert np.array_equal(gm["LeftIndex"], w_idx.astype(np.uint32))
    g, e = got["distance"][0][w_idx], exp["distance"][0]
    if p.distance_kind == _abi.DIST_PINHOLE:
        assert g.tobytes() == e.tobytes()
    else:
        assert np.array_equal(np.isinf(g), np.isinf(e)) and np.allclose(g[np.isfinite(e)], e[np.isfinite(e)], rtol=1e-12, atol=0)
        ok = gm["RightIndex"] != _abi.NO_MATCH
        d = got["disparity_u16"][0][w_idx][ok]
        assert g[ok].tobytes() == ctx.distance_lut(p.distance_kind, f.width)[d].tobytes()
        assert (g[~ok] == 0.0).all()


# The dense SAD key packs cost << xb | code below bit 31, xb = ceil_log2(nxc + 33) (usv_dense.cu). 32x64 gray: the
# largest cost 255 * 2048 needs 19 bits, so xb <= 12 and nxc <= 4063: width 4094. 32x32 colour: 255 * 3072 needs 20
# bits, xb <= 11, nxc <= 2015: width 2046. One pixel wider, the gray SAD and colour SAD arms of the ALU correlation
# kernel take the job.
KEY_CASES = [(1, 64, 4094, "dense_sad_argmin_kernel"), (1, 64, 4095, "dense_corr_argmin_kernel"),
             (3, 32, 2046, "dense_sad_argmin_kernel"), (3, 32, 2047, "dense_corr_argmin_kernel")]


@pytest.mark.gpu
@pytest.mark.parametrize("pat", PATTERNS)
@pytest.mark.parametrize("c,th,w,kernel", KEY_CASES)
def test_dense_sad_key_limit(ctx, oracle, c, th, w, kernel, pat):
    left, right = pattern(pat, 1, th + 3, w, c, seed=w)
    p = _abi.make_params(tmpl_w=32, tmpl_h=th, cost="sad", search_max=255, accept_threshold=ACCEPT_ALL)
    got, name = _run_dense(ctx, left, right, p, INT_MASK | _abi.OUT_DISTANCE)
    assert name == kernel
    exp = reference_dense(left, right, p)
    _compare(got, exp, _abi.COST_SAD, "%s w=%d" % (pat, w))
    _check_sampled(ctx, oracle, got, left, right, p, 250, seed=w)
    if pat == "saturated":
        assert (got["raw_cost"] == 255 * 32 * th * c).all()
        nxc = w - 31
        assert np.array_equal(got["right_index"][0] % nxc, np.maximum(np.arange(nxc) - 255, 0)[None, :].repeat(4, 0).ravel())


# Sab of a 32768-byte template is at most 65025 * 32768 = 2 130 739 200 < 2^31 (the s32 accumulators of both
# tensor-pipe kernels); on the "full" frames every window and candidate has exactly that Sab (32x341x3: 2 128 658 400).
# tcgen05 keeps running sums E (rows that entered the band) and L (rows that left) and caps the band height at
# (2^31 - 1) / (65025 * 32 * C) - th rows (usv_dense_umma.cu): 8 rows for 32x1024 gray, 3 rows for 32x341 colour. The
# output rows are a multiple of the cap (24 and 21), so the bands are exactly that tall and, on the "full" frames, E
# reaches its largest value: th + bh - 1 rows of 65025 * 32 * C, i.e. 1031 * 2 080 800 = 2 145 304 800 (gray) and
# 343 * 6 242 400 = 2 141 143 200 (colour).
S32_OUT_ROWS = {1: 24, 3: 21}


@pytest.mark.gpu
@pytest.mark.parametrize("pat", PRODUCT_PATTERNS)
@pytest.mark.parametrize("cost", ["ncc", "zncc", "ssd"])
@pytest.mark.parametrize("c,th", [(1, 1024), (3, 341)])
def test_tensor_pipe_s32_sums(ctx, oracle, c, th, cost, pat):
    nyc = S32_OUT_ROWS[c]
    left, right = pattern(pat, 1, th + nyc - 1, 300, c, seed=th)
    p = _abi.make_params(tmpl_w=32, tmpl_h=th, cost=cost, search_max=127, accept_threshold=ACCEPT_ALL)
    exp = reference_dense(left, right, p)
    if pat == "full":  # every candidate ties: SSD 0, NCC one value, ZNCC 0 (zero variance); the first candidate wins
        if cost == "ssd":
            assert (exp["raw_cost"] == 0).all()
        else:
            assert len(np.unique(exp["score"])) == 1
        assert np.array_equal(exp["right_index"][0] % 269, np.tile(np.maximum(np.arange(269) - 127, 0), nyc))
    for kernel, name in (("mma", "dense_corr_mma_kernel"), ("tcgen05", "dense_corr_umma_kernel")):
        got, used = _run_dense(ctx, left, right, p, _mask(cost) | _abi.OUT_RAW_COST | _abi.OUT_DISTANCE, kernel)
        assert used == name
        _compare(got, exp, _abi.COST_NAMES[cost], "%s %s" % (kernel, pat))
        _check_sampled(ctx, oracle, got, left, right, p, 60, seed=c)
    if pat == "dips" and cost != "ssd":
        d = exp["disparity_u16"][0].reshape(nyc, 269)[:, SHIFT:]
        assert (d == SHIFT).mean() > 0.9


# mma.sync scores SSD in u32 when 65025 * n < 2^28 (32x129: 268 423 200), with 2^30 marking out-of-frame columns; 32x130
# takes the f64 path. search_max 255 on a 300-px frame clips the range of most windows at the frame's edge.
@pytest.mark.gpu
@pytest.mark.parametrize("pat", PATTERNS)
@pytest.mark.parametrize("side", [_abi.LEFT_CAM, _abi.RIGHT_CAM])
@pytest.mark.parametrize("th", [129, 130])
def test_mma_ssd_u32_limit(ctx, oracle, th, side, pat):
    left, right = pattern(pat, 1, th + 11, 300, 1, camera_side=side, seed=th)
    p = _abi.make_params(tmpl_w=32, tmpl_h=th, cost="ssd", camera_side=side, search_max=255, accept_threshold=ACCEPT_ALL,
                         distance_kind=_abi.DIST_POWERLAW)
    got, name = _run_dense(ctx, left, right, p, INT_MASK | _abi.OUT_DISTANCE, "mma")
    assert name == "dense_corr_mma_kernel"
    _compare(got, reference_dense(left, right, p), _abi.COST_SSD, pat)
    _check_sampled(ctx, oracle, got, left, right, p, 200, seed=th + side)


def _host_error_code(fn):
    with pytest.raises(api.UsvError) as e:
        fn()
    return str(e.value)


@pytest.mark.gpu
def test_raw_cost_u16_stays_below_its_sentinel(ctx):
    """255 * n must stay below 0xFFFF, the "no candidate" value: n = 256 passes with its largest cost 65280, n = 257
    (whose saturated cost would be 65535) is refused for dense and sparse calls alike."""
    mask = _abi.OUT_RAW_COST | _abi.OUT_RAW_COST_U16 | _abi.OUT_RIGHT_INDEX
    left, right = pattern("saturated", 1, 20, 60, 1)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_min=3, search_max=40, accept_threshold=ACCEPT_ALL)
    got = ctx.match_dense(left, right, p, mask=mask)
    assert ctx.last_kernel == "dense_sad_argmin_kernel"
    has = got["raw_cost"] != 0xFFFFFFFF
    assert (got["raw_cost"][has] == 65280).all() and (got["raw_cost_u16"][~has] == 0xFFFF).all() and (~has).any()
    assert np.array_equal(got["raw_cost_u16"][has], got["raw_cost"][has].astype(np.uint16))
    gs = ctx.match_templates(left, right, [0, 10, 44], [0, 2, 4], p, mask=mask)
    assert ctx.last_kernel == "block_cost_argmin_direct"
    assert gs["raw_cost_u16"].tolist() == [[0xFFFF, 65280, 65280]]
    for tw, th in ((257, 1), (1, 257)):
        q = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="sad", search_max=40)
        lf, rt = pattern("saturated", 1, th + 2, tw + 20, 1)
        assert "(-4)" in _host_error_code(lambda: ctx.match_dense(lf, rt, q, mask=mask))
        assert "(-4)" in _host_error_code(lambda: ctx.match_templates(lf, rt, [5], [0], q, mask=mask))


def _resolved_expected(oracle, winners, disparity):
    alive = np.zeros(len(winners), bool)
    kept = oracle.resolve_match_list(winners[winners["RightIndex"] != _abi.NO_MATCH])
    alive[np.unique(kept["LeftIndex"])] = True
    return np.where(alive, disparity, _abi.NO_DISPARITY).astype(np.uint16)


@pytest.mark.gpu
@pytest.mark.parametrize("cost", ["sad", "zncc"])
def test_resolved_rows_at_2048_windows(ctx, oracle, cost):
    """nx = 2048 windows per row (width 2047 + tw) is the widest row the resolve kernel serves; flat rows make whole
    buckets of windows claim the same candidate with the same value. One pixel wider is refused."""
    tw = 16
    left, right = pattern("dips", 1, tw + 5, 2047 + tw, 1, seed=1)
    left[:, :tw + 2], right[:, :tw + 2] = 90, 90
    p = _abi.make_params(tmpl_w=tw, tmpl_h=tw, cost=cost, search_max=255, accept_threshold=ACCEPT_ALL)
    assert api.grid_dims(_abi.frame_desc_for(left), p)[0] == 2048
    got = ctx.match_dense(left, right, p, mask=_mask(cost) | _abi.OUT_RESOLVED_DISPARITY_U16)
    assert ctx.last_kernel == {"sad": "dense_sad_argmin_kernel", "zncc": "dense_corr_umma_kernel"}[cost]
    exp = reference_dense(left, right, p)
    _compare(got, exp, _abi.COST_NAMES[cost], "winners")
    assert np.array_equal(got["resolved_disparity_u16"][0], _resolved_expected(oracle, exp["matches"][0], exp["disparity_u16"][0]))
    lf, rt = pattern("dips", 1, tw + 5, 2048 + tw, 1, seed=1)
    assert "(-4)" in _host_error_code(lambda: ctx.match_dense(lf, rt, p, mask=_abi.OUT_RESOLVED_DISPARITY_U16))


def _templates_host(ctx, left, right, tx, ty, p, row_cap, mask):
    """usv_match_templates_host with a caller-chosen row_cap (the Python wrapper always passes the frame width)."""
    f = _abi.frame_desc_for(left)
    n, nt = left.shape[0], len(tx)
    tx, ty = np.ascontiguousarray(tx, np.int32), np.ascontiguousarray(ty, np.int32)
    arrs, st = api._alloc_host_outputs(n * nt, mask)
    integer = p.cost_kind <= _abi.COST_SSD
    cost_rows = np.full((n, nt, row_cap), 0xFFFFFFFF, np.uint32) if integer else None
    score_rows = np.full((n, nt, row_cap), np.nan) if not integer else None
    rc = api.lib().usv_match_templates_host(ctx._h, api._ptr(left), api._ptr(right), C.byref(f), C.c_int32(n), api._ptr(tx),
                                            api._ptr(ty), C.c_int32(nt), C.byref(p), C.byref(st), api._ptr(cost_rows),
                                            api._ptr(score_rows), C.c_int32(row_cap))
    ctx._check(rc, "usv_match_templates_host")
    out = {k: v.reshape(n, nt) for k, v in arrs.items()}
    out["rows"] = cost_rows if integer else score_rows
    return out


def _check_sparse(got, left, right, tx, ty, p, row_cap=None):
    integer = p.cost_kind <= _abi.COST_SSD
    nxc = left.shape[2] - p.tmpl_w + 1
    for i, (x, y) in enumerate(zip(tx, ty)):
        xr, v = reference_candidates(left, right, int(x), int(y), p)
        if integer:
            j = int(np.argmin(v)) if len(v) else -1
            assert got["raw_cost"][0, i] == (v[j] if j >= 0 else 0xFFFFFFFF), (x, y)
        else:
            j = int(np.argmin(1.0 - v)) if len(v) else -1
            assert got["score"][0, i].tobytes() == (np.float64(v[j]) if j >= 0 else np.float64(0.0)).tobytes(), (x, y)
        assert got["right_index"][0, i] == (y * nxc + xr[j] if j >= 0 else _abi.NO_MATCH), (x, y)
        if row_cap is not None:
            k = min(len(v), row_cap)
            rows = got["rows"][0, i]
            assert rows[:k].tobytes() == v[:k].astype(rows.dtype).tobytes(), (x, y)
            untouched = rows[k:]
            assert (untouched == 0xFFFFFFFF).all() if integer else np.isnan(untouched).all()


# The direct form stages strips of at most 64 KB, so a 32-px template on a frame of 544 px or more (512 candidates +
# 32 px per pass) gets fewer strip rows than template rows: 32x64 colour about 39 rows, 32x1024 gray about 113.
@pytest.mark.gpu
@pytest.mark.parametrize("cost", ["sad", "zncc"])
@pytest.mark.parametrize("c,th", [(3, 64), (1, 1024)])
def test_direct_row_chunked_strips(ctx, oracle, c, th, cost):
    w = 560
    left, right = pattern("dips", 1, th + 6, w, c, seed=th)
    nxc, nyc = w - 31, 7
    rng = np.random.default_rng(th)
    tx = np.r_[0, 1, nxc - 1, 255, 256, rng.integers(0, nxc, 20)].astype(np.int32)
    ty = np.r_[0, nyc - 1, 3, 0, nyc - 1, rng.integers(0, nyc, 20)].astype(np.int32)
    p = _abi.make_params(tmpl_w=32, tmpl_h=th, cost=cost, search_max=255, accept_threshold=ACCEPT_ALL)
    got = _templates_host(ctx, left, right, tx, ty, p, 100, _mask(cost) | _abi.OUT_RAW_COST)
    assert ctx.last_kernel == "block_cost_argmin_direct"
    _check_sparse(got, left, right, tx, ty, p, row_cap=100)
    if c == 1 and cost == "sad":  # the dense sweep of this shape falls back to the direct form as well (th > 64)
        got, name = _run_dense(ctx, left, right, p, INT_MASK | _abi.OUT_DISTANCE)
        assert name == "block_cost_argmin_direct"
        _compare(got, reference_dense(left, right, p), _abi.COST_SAD, "dense")
        _check_sampled(ctx, oracle, got, left, right, p, 40)


@pytest.mark.gpu
@pytest.mark.parametrize("cost", ["sad", "zncc"])
@pytest.mark.parametrize("tw", [1, 4, 8, 16, 32, 64, 256])
def test_template_envelope_runs_or_is_refused(ctx, tw, cost):
    """Every template shape the validation accepts (up to 32768 bytes, rows up to 1024 bytes) either runs and matches the
    reference or is refused with USV_ERR_UNSUPPORTED, for dense and sparse calls: never a failed launch."""
    th = 32768 // tw
    left, right = pattern("dips", 1, th + 1, tw + 7, 1, seed=tw)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost=cost, search_min=-2, search_max=5, accept_threshold=ACCEPT_ALL)
    ran = []
    try:
        got = ctx.match_dense(left, right, p, mask=_mask(cost) | _abi.OUT_RAW_COST)
        ran.append(ctx.last_kernel)
        _compare(got, reference_dense(left, right, p), _abi.COST_NAMES[cost], "dense")
    except api.UsvError as e:
        assert "(-4)" in str(e), str(e)
    tx, ty = np.array([0, 3, 7, 7], np.int32), np.array([0, 1, 0, 1], np.int32)
    try:
        got = _templates_host(ctx, left, right, tx, ty, p, 4, _mask(cost) | _abi.OUT_RAW_COST)
        ran.append(ctx.last_kernel)
        _check_sparse(got, left, right, tx, ty, p, row_cap=4)
    except api.UsvError as e:
        assert "(-4)" in str(e), str(e)
    if tw >= 16:  # the direct form holds these whole
        assert "block_cost_argmin_direct" in ran


# ---- dirty padding ----------------------------------------------------------------------------------------------------
# name: (channels, params, corr_kernel, kernel, sparse, extra outputs)
DIRTY = {
    "sad_gray": (1, dict(tmpl_w=16, tmpl_h=16, cost="sad"), "auto", "dense_sad_argmin_kernel", False, 0),
    "sad_colour": (3, dict(tmpl_w=16, tmpl_h=16, cost="sad"), "auto", "dense_sad_argmin_kernel", False, 0),
    "alu_zncc": (1, dict(tmpl_w=12, tmpl_h=10, cost="zncc"), "alu", "dense_corr_argmin_kernel", False, 0),
    "alu_ssd_colour": (3, dict(tmpl_w=16, tmpl_h=8, cost="ssd"), "alu", "dense_corr_argmin_kernel", False, 0),
    "alu_sad_colour": (3, dict(tmpl_w=12, tmpl_h=8, cost="sad"), "alu", "dense_corr_argmin_kernel", False, 0),
    "mma_ssd": (1, dict(tmpl_w=32, tmpl_h=12, cost="ssd"), "mma", "dense_corr_mma_kernel", False, 0),
    "mma_zncc_colour": (3, dict(tmpl_w=13, tmpl_h=9, cost="zncc"), "mma", "dense_corr_mma_kernel", False, 0),
    "tcgen05_ncc": (1, dict(tmpl_w=16, tmpl_h=16, cost="ncc"), "tcgen05", "dense_corr_umma_kernel", False, 0),
    "tcgen05_zncc_colour": (3, dict(tmpl_w=32, tmpl_h=7, cost="zncc"), "tcgen05", "dense_corr_umma_kernel", False, 0),
    "direct_sad": (1, dict(tmpl_w=7, tmpl_h=5, cost="sad"), "auto", "block_cost_argmin_direct", False, 0),
    "direct_zncc_colour": (3, dict(tmpl_w=40, tmpl_h=4, cost="zncc"), "auto", "block_cost_argmin_direct", False, 0),
    "sparse_ssd": (1, dict(tmpl_w=13, tmpl_h=6, cost="ssd"), "auto", "block_cost_argmin_direct", True, 0),
    "sparse_ncc_colour": (3, dict(tmpl_w=16, tmpl_h=16, cost="ncc"), "auto", "block_cost_argmin_direct", True, 0),
    "resolve_rows": (1, dict(tmpl_w=16, tmpl_h=16, cost="sad"), "auto", "dense_sad_argmin_kernel", False,
                     _abi.OUT_RESOLVED_DISPARITY_U16),
}
DIRTY_CASES = [(name, w) for name, cfg in DIRTY.items() for w in ((97, 131) if cfg[0] == 1 else (97,))]
H, N = 40, 2


def _dirty_copy(frames, row_stride, frame_stride, fill, rng):
    """frames [n, H, W(, C)] written into a buffer of the given layout whose padding and gaps hold `fill` (a byte, or
    "random"); returns (buffer, view [n, H, W(, C)] on it)."""
    n, h = frames.shape[:2]
    rb = frames[0, 0].size
    total = (n - 1) * frame_stride + h * row_stride
    buf = rng.integers(0, 256, total, dtype=np.uint8) if fill == "random" else np.full(total, fill, np.uint8)
    view = np.lib.stride_tricks.as_strided(buf, shape=frames.shape, strides=(frame_stride, row_stride) + frames.strides[2:])
    view[...] = frames
    pad = np.lib.stride_tricks.as_strided(buf[rb:], shape=(n, h, row_stride - rb), strides=(frame_stride, row_stride, 1))
    assert (pad != 0).any() and (fill == "random" or (pad == fill).all())
    if frame_stride > h * row_stride:
        assert (buf[h * row_stride:frame_stride] != 0).any()
    return buf, view


def _dirty_expected(oracle, left, right, p, mask, sparse, tx, ty):
    if sparse:
        return oracle.match_templates(left, right, tx, ty, p, mask=mask & ~_abi.OUT_RESOLVED_DISPARITY_U16)
    exp = oracle.match_dense(left, right, p, mask=(mask | _abi.OUT_MATCHES) & ~_abi.OUT_RESOLVED_DISPARITY_U16)
    if mask & _abi.OUT_RESOLVED_DISPARITY_U16:
        exp["resolved_disparity_u16"] = np.stack([_resolved_expected(oracle, exp["matches"][i], exp["disparity_u16"][i])
                                                  for i in range(len(left))])
    return exp


def _device_run(ctx, left, right, p, mask, sparse, tx, ty, fill, rng):
    torch = pytest.importorskip("torch")
    rb = left[0, 0].size
    row_stride = (rb + 16) & ~15 if rb % 16 else rb + 32  # always some padding, 16-byte aligned
    frame_stride = H * row_stride + 48
    dl = torch.from_numpy(_dirty_copy(left, row_stride, frame_stride, fill, rng)[0]).cuda()
    dr = torch.from_numpy(_dirty_copy(right, row_stride, frame_stride, fill, rng)[0]).cuda()
    f = _abi.FrameDesc(left.shape[2], H, left[0, 0, 0].size, row_stride, frame_stride)
    n_win = len(tx) if sparse else api.grid_dims(f, p)[0] * api.grid_dims(f, p)[1]
    outs, st = {}, _abi.Outputs()
    for name, bit, dt in _abi.OUTPUT_FIELDS:
        if mask & bit:
            outs[name] = torch.zeros(N * n_win * dt.itemsize, dtype=torch.uint8, device="cuda")
            setattr(st, name, outs[name].data_ptr())
    stream = torch.cuda.current_stream().cuda_stream
    if sparse:
        dtx, dty = torch.from_numpy(tx).cuda(), torch.from_numpy(ty).cuda()
        ctx.match_templates_device(dl.data_ptr(), dr.data_ptr(), f, N, dtx.data_ptr(), dty.data_ptr(), len(tx), p, st, stream)
    else:
        ctx.match_dense_device(dl.data_ptr(), dr.data_ptr(), f, N, p, st, stream)
    torch.cuda.synchronize()
    assert api.lib().usv_device_status(ctx._h) == 0
    dts = {name: dt for name, _, dt in _abi.OUTPUT_FIELDS}
    return {k: v.cpu().numpy().view(dts[k]).reshape(N, n_win) for k, v in outs.items()}


def _stream_run(ctx, left, right, p, mask, gather, fill, rng):
    w, c = left.shape[2], left[0, 0, 0].size
    st = ctx.stream(_abi.FrameDesc(w, H, c, w * c, w * c * H), p, pairs_per_slot=N, n_slots=1, mask=mask)
    try:
        f = st.frame
        assert f.row_stride % 128 == 0 and f.row_stride > w * c
        _, lv = _dirty_copy(left, f.row_stride, f.frame_stride, fill, rng)
        _, rv = _dirty_copy(right, f.row_stride, f.frame_stride, fill, rng)
        if gather:  # pairs in reverse store order
            st.submit_gather(0, lv, [1, 0], rv, [1, 0])
        else:
            st.submit_from(0, lv, rv)
        st.wait(0)
        out = {k: v.copy() for k, v in st.slots[0]["out"].items()}
    finally:
        st.close()
    return {k: v[::-1] for k, v in out.items()} if gather else out


def _host_run(ctx, left, right, p, mask, sparse, tx, ty):
    w, c = left.shape[2], left[0, 0, 0].size
    pitch = (w * c + 127) & ~127
    primer = np.full((N, H + 3, pitch // c) + ((c,) if c > 1 else ()), 255, np.uint8)
    assert primer[0, 0].size == pitch  # the host path's staging pitch: every byte of it now holds 255
    if sparse:
        ctx.match_templates(primer, primer, tx, ty, p, mask=_abi.OUT_RIGHT_INDEX)
        return ctx.match_templates(left, right, tx, ty, p, mask=mask)
    ctx.match_dense(primer, primer, p, mask=_abi.OUT_RIGHT_INDEX)
    return ctx.match_dense(left, right, p, mask=mask)


@pytest.mark.gpu
@pytest.mark.parametrize("name,w", DIRTY_CASES)
def test_dirty_padding(ctx, oracle, name, w):
    c, kw, kernel, expect, sparse, extra = DIRTY[name]
    left, right = synth.make_pairs(N, w, H, c, shift=9, noise_sigma=2.0, seed=w + c)
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    p = _abi.make_params(search_max=40, accept_threshold=ACCEPT_ALL, **kw)
    kind = p.cost_kind
    mask = (INT_MASK if kind <= _abi.COST_SSD else FLOAT_MASK) | extra
    nxc, nyc = w - p.tmpl_w + 1, H - p.tmpl_h + 1
    tx = np.array([0, nxc - 1, nxc // 2, 5, nxc - 2], np.int32)
    ty = np.array([0, nyc - 1, nyc // 2, nyc - 1, 0], np.int32)
    exp = _dirty_expected(oracle, left, right, p, mask, sparse, tx, ty)
    rng = np.random.default_rng(w)
    ctx.corr_kernel(kernel)
    try:
        for fill in (0xFF, "random"):
            got = _device_run(ctx, left, right, p, mask, sparse, tx, ty, fill, rng)
            assert ctx.last_kernel == expect
            _compare(got, exp, kind, "device %s" % fill)
            if extra:
                assert np.array_equal(got["resolved_disparity_u16"], exp["resolved_disparity_u16"])
            if sparse:
                continue
            for gather in (False, True):
                got = _stream_run(ctx, left, right, p, mask, gather, fill, rng)
                assert ctx.last_kernel == expect
                _compare(got, exp, kind, "stream gather=%s %s" % (gather, fill))
                if extra:
                    assert np.array_equal(got["resolved_disparity_u16"], exp["resolved_disparity_u16"])
        got = _host_run(ctx, left, right, p, mask, sparse, tx, ty)
        assert ctx.last_kernel == expect
        _compare(got, exp, kind, "host")
    finally:
        ctx.corr_kernel("auto")
