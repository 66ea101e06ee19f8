"""GPU parity: the CUDA path, called through the C-ABI, against the CPU oracle on
the same seeded inputs and against the committed golden fixtures.

Bar: bit-exact for integer costs, indices, disparities, Match records and (for
NCC/ZNCC) the f64 scores, which are computed from exact integer sums with the
same IEEE operations as the oracle. Distances: <= 1e-12 relative (device pow vs
libm pow; the north-star tolerance is 1e-3)."""
import os

import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
DIST_RTOL = 1e-12


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def assert_same(got, exp, float_kind):
    for k in ("right_index", "raw_cost", "disparity_u16"):
        assert np.array_equal(got[k], exp[k]), k
    assert np.array_equal(got["matches"]["LeftIndex"], exp["matches"]["LeftIndex"])
    assert np.array_equal(got["matches"]["RightIndex"], exp["matches"]["RightIndex"])
    # MatchValue / score: bit-exact (inf == inf included)
    assert got["matches"]["MatchValue"].tobytes() == exp["matches"]["MatchValue"].tobytes()
    assert got["score"].tobytes() == exp["score"].tobytes()
    for k in ("distance", "distance_f32"):
        g, e = got[k].astype(np.float64), exp[k].astype(np.float64)
        assert np.array_equal(np.isinf(g), np.isinf(e)) and np.array_equal(np.isnan(g), np.isnan(e)), k
        fin = np.isfinite(e)
        tol = DIST_RTOL if k == "distance" else 1e-6
        assert np.allclose(g[fin], e[fin], rtol=tol, atol=0), k


def _golden_cases():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.CASES


CASES = _golden_cases()


@pytest.mark.parametrize("name", sorted(CASES))
def test_dense_vs_golden(ctx, name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    kw = CASES[name][5]
    p = _abi.make_params(**kw)
    got = ctx.match_dense(z["left"], z["right"], p)
    exp = {k[4:]: z[k] for k in z.files if k.startswith("out_")}
    assert_same(got, exp, kw["cost"] in ("ncc", "zncc"))


SWEEP = [
    # W, H, C, shift, params
    (640, 40, 1, 37, dict(tmpl_w=16, tmpl_h=16, cost="sad")),                                   # C2 geometry, thin band
    (640, 36, 1, 37, dict(tmpl_w=16, tmpl_h=16, cost="sad", search_max=127)),                   # D=128 variant
    (640, 36, 1, 37, dict(tmpl_w=16, tmpl_h=16, cost="ssd", search_max=127)),
    (320, 40, 3, 20, dict(tmpl_w=32, tmpl_h=32, cost="zncc", search_max=255, accept_threshold=0.4)),  # C3 geometry, cropped
    (320, 40, 3, 20, dict(tmpl_w=32, tmpl_h=32, cost="ncc", search_max=63)),
    (200, 30, 1, -15, dict(tmpl_w=16, tmpl_h=16, cost="sad", camera_side=_abi.RIGHT_CAM, search_max=64)),
    (131, 29, 1, 9, dict(tmpl_w=7, tmpl_h=5, cost="sad", search_min=1, search_max=33)),          # ragged sizes
    (131, 29, 2, 9, dict(tmpl_w=5, tmpl_h=3, cost="ssd", search_max=20)),                        # row bytes not /4
    (77, 23, 4, 4, dict(tmpl_w=9, tmpl_h=9, cost="zncc", search_max=30, distance_kind=_abi.DIST_POWERLAW)),
    (96, 33, 3, 6, dict(tmpl_w=11, tmpl_h=4, cost="sad", stride_x=2, stride_y=3, search_max=40)),
    (64, 64, 1, 5, dict(tmpl_w=64, tmpl_h=64, cost="ssd")),                                      # one window, max template
    (600, 24, 1, 3, dict(tmpl_w=16, tmpl_h=16, cost="sad", search_min=-8, search_max=8)),         # signed range
    (400, 30, 1, 21, dict(tmpl_w=8, tmpl_h=8, cost="sad", search_max=90)),                        # dense kernel, 2-word windows
    (400, 30, 1, 21, dict(tmpl_w=12, tmpl_h=9, cost="sad", search_max=90)),                       # 3-word windows
    (400, 40, 1, 21, dict(tmpl_w=24, tmpl_h=24, cost="sad")),                                     # 6-word windows, full range
    (400, 40, 1, -21, dict(tmpl_w=32, tmpl_h=20, cost="sad", camera_side=_abi.RIGHT_CAM)),         # 8-word windows, RightCam
]


@pytest.mark.parametrize("w,h,c,shift,kw", SWEEP)
def test_dense_vs_oracle(ctx, oracle, w, h, c, shift, kw):
    left, right = synth.make_pairs(2, w, h, c, shift=shift, noise_sigma=2.0, seed=w * 7 + h)
    p = _abi.make_params(**kw)
    got = ctx.match_dense(left, right, p)
    exp = oracle.match_dense(left, right, p)
    assert_same(got, exp, kw["cost"] in ("ncc", "zncc"))
    assert ctx.launch_count > 0


@pytest.mark.parametrize("kind", ["sad", "ssd", "ncc", "zncc"])
def test_templates_full_cost_rows(ctx, oracle, kind):
    """Config C1: single 640x480 pair, shift 37, one 16x16 template at (300, 200),
    full-row search — every candidate's cost, not only the winner."""
    left, right = synth.make_pairs(1, 640, 480, 1, shift=37, noise_sigma=2.0, seed=325)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost=kind)
    tx, ty = [300, 0, 624, 37], [200, 0, 464, 100]
    got = ctx.match_templates(left, right, tx, ty, p, rows=True)
    exp = oracle.match_templates(left, right, tx, ty, p, rows=True)
    assert_same(got, exp, kind in ("ncc", "zncc"))
    if kind in ("sad", "ssd"):
        assert np.array_equal(got["cost_rows"], exp["cost_rows"])
    else:
        assert got["score_rows"].tobytes() == exp["score_rows"].tobytes()
    assert got["disparity_u16"][0, 0] == 37  # the known shift is recovered


def test_tie_break_flat_frames(ctx, oracle):
    left = np.full((1, 24, 128), 9, np.uint8)
    for side in (_abi.LEFT_CAM, _abi.RIGHT_CAM):
        for kind in ("sad", "zncc"):
            p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost=kind, camera_side=side, search_max=50, accept_threshold=2.0)
            got = ctx.match_dense(left, left.copy(), p)
            exp = oracle.match_dense(left, left.copy(), p)
            assert_same(got, exp, kind == "zncc")


def test_empty_ranges_and_threshold(ctx, oracle):
    left, right = synth.make_pairs(1, 80, 20, 1, shift=3, noise_sigma=30.0, seed=2)
    for kw in (dict(search_min=10, search_max=12), dict(search_min=0, search_max=6, accept_threshold=0.02)):
        p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="sad", **kw)
        got = ctx.match_dense(left, right, p)
        exp = oracle.match_dense(left, right, p)
        assert_same(got, exp, False)
        assert (got["right_index"] == _abi.NO_MATCH).any()


def test_unaligned_host_stride(ctx, oracle):
    """Host frames with an odd row stride go through the repacking H2D path."""
    rng = np.random.default_rng(4)
    buf_l = rng.integers(0, 256, (2, 30, 101), dtype=np.uint8)
    buf_r = rng.integers(0, 256, (2, 30, 101), dtype=np.uint8)
    left, right = buf_l[:, :, :97], buf_r[:, :, :97]
    p = _abi.make_params(tmpl_w=12, tmpl_h=12, cost="ssd", search_max=30)
    got = ctx.match_dense(left, right, p)
    exp = oracle.match_dense(np.ascontiguousarray(left), np.ascontiguousarray(right), p)
    assert_same(got, exp, False)


def test_invalid_arguments_fail_loudly(ctx):
    left, right = synth.make_pairs(1, 64, 32, 1)
    with pytest.raises(api.UsvError):
        ctx.match_dense(left, right, _abi.make_params(tmpl_w=128, tmpl_h=8))
    with pytest.raises(api.UsvError):
        ctx.match_dense(left, right, _abi.make_params(tmpl_w=8, tmpl_h=8, cost=7))
    with pytest.raises(api.UsvError):
        ctx.match_templates(left, right, [60], [0], _abi.make_params(tmpl_w=8, tmpl_h=8))


# ---- distance family ---------------------------------------------------------
def test_disparity_to_distance(ctx, oracle):
    d = np.arange(-3, 700, dtype=np.int32)
    for kind in (_abi.DIST_PINHOLE, _abi.DIST_POWERLAW):
        got = ctx.disparity_to_distance(d, kind)
        exp = oracle.distance(d, kind)
        assert np.array_equal(np.isnan(got), np.isnan(exp)) and np.array_equal(np.isinf(got), np.isinf(exp))
        fin = np.isfinite(exp)
        assert np.allclose(got[fin], exp[fin], rtol=DIST_RTOL, atol=0)
    assert ctx.disparity_to_distance([40], _abi.DIST_POWERLAW)[0] == pytest.approx(556.401951467, rel=1e-11)


MS = 1_000_000


def test_moving_object_distance(ctx, oracle):
    args = (110 * MS, [(300, 200)], [(260, 200)], [(250, 200)], [(240, 200)], [(0, 0, 0)], 100 * MS, 67 * MS, 33 * MS)
    assert ctx.moving_object_distance(1, *args)[0] == pytest.approx(626.463714398, rel=1e-11)
    rng = np.random.default_rng(7)
    for trial in range(100):
        n_other, n_old, n_older = (int(rng.integers(0 if trial % 10 == 0 else 1, 6)) for _ in range(3))
        n_idx, n_this = int(rng.integers(0, 8)), int(rng.integers(0, 8))
        t_older = int(rng.integers(0, 10**9))
        t_old = t_older + int(rng.integers(0 if trial % 7 == 0 else 1, 50 * MS))  # zero gaps -> inf / NaN paths
        t_other = t_old + int(rng.integers(1, 50 * MS))
        t_this = t_other + int(rng.integers(-20 * MS, 20 * MS))
        a = (t_this, rng.uniform(0, 640, (n_this, 2)), rng.uniform(0, 640, (n_other, 2)), rng.uniform(0, 640, (n_old, 2)),
             rng.uniform(0, 640, (n_older, 2)), rng.integers(-1, 7, (n_idx, 3)), t_other, t_old, t_older)
        for side in (0, 1):
            got = ctx.moving_object_distance(side, *a)
            exp = oracle.moving_object_distance(side, *a)
            assert got.shape == exp.shape
            assert np.array_equal(np.isnan(got), np.isnan(exp)) and np.array_equal(np.isinf(got), np.isinf(exp)), trial
            fin = np.isfinite(exp)
            assert np.allclose(got[fin], exp[fin], rtol=DIST_RTOL, atol=0), trial


def test_coordinate_position(ctx, oracle):
    for side, exp in ((1, (9.103702, 99.584751, 12.454575)), (0, (-18.505677, 98.272783, 8.532612))):
        assert ctx.coordinate_position(side, [100.0], [(300, 200)])[0] == pytest.approx(exp, abs=1e-6)
    rng = np.random.default_rng(3)
    dist = rng.uniform(15, 2000, 500)
    xy = np.stack([rng.uniform(0, 640, 500), rng.uniform(0, 480, 500)], 1)
    for side in (0, 1):
        got = ctx.coordinate_position(side, dist, xy)
        exp = oracle.coordinate_position(side, dist, xy)
        assert np.array_equal(np.isnan(got), np.isnan(exp))
        fin = np.isfinite(exp)
        assert np.allclose(got[fin], exp[fin], rtol=1e-9, atol=1e-9)


# ---- streamed path -------------------------------------------------------------
def test_stream_matches_oracle(ctx, oracle):
    w, h = 160, 40
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_max=63)
    f = _abi.FrameDesc(w, h, 1, w, w * h)
    mask = _abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST | _abi.OUT_DISTANCE_F32 | _abi.OUT_DISPARITY_U16
    st = ctx.stream(f, p, pairs_per_slot=3, n_slots=2, mask=mask)
    left, right = synth.make_pairs(7, w, h, 1, shift=11, noise_sigma=2.0, seed=8)
    exp = oracle.match_dense(left, right, p)
    batches = [(0, 3), (3, 6), (6, 7)]
    pending = []
    for bi, (a, b) in enumerate(batches):
        slot = bi % 2
        if len(pending) == 2:
            s0, a0, b0 = pending.pop(0)
            st.wait(s0)
            for k in ("right_index", "raw_cost", "disparity_u16"):
                assert np.array_equal(st.slots[s0]["out"][k][: b0 - a0], exp[k][a0:b0]), k
        st.slots[slot]["left"][: b - a] = left[a:b]
        st.slots[slot]["right"][: b - a] = right[a:b]
        st.submit(slot, b - a)
        pending.append((slot, a, b))
    for s0, a0, b0 in pending:
        st.wait(s0)
        for k in ("right_index", "raw_cost", "disparity_u16"):
            assert np.array_equal(st.slots[s0]["out"][k][: b0 - a0], exp[k][a0:b0]), k
        assert np.allclose(st.slots[s0]["out"]["distance_f32"][: b0 - a0], exp["distance_f32"][a0:b0], rtol=1e-6)
    assert st.h2d_bytes_per_pair == 2 * 256 * h and st.d2h_bytes_per_pair == (4 + 4 + 4 + 2) * st.nx * st.ny
    st.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cost,c", [("zncc", 3), ("ssd", 1), ("zncc", 1)])  # the last one: concurrent tcgen05 kernels (TMEM allocation across streams)
def test_stream_slots_do_not_share_scratch(ctx, oracle, cost, c):
    """The sliding correlation kernel keeps planes and window statistics in a scratch buffer; slots of a stream run
    concurrently on their own CUDA streams and must each own one (several batches in flight, then compare)."""
    w, h, n_slots, pps = 200, 60, 4, 2
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost=cost, search_max=63)
    left, right = synth.make_pairs(n_slots * pps * 2, w, h, c, shift=11, noise_sigma=2.0, seed=21)
    exp = oracle.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX)
    st = ctx.stream(_abi.frame_desc_for(left), p, pairs_per_slot=pps, n_slots=n_slots, mask=_abi.OUT_RIGHT_INDEX)
    for rnd in range(2):
        for s in range(n_slots):
            a = (rnd * n_slots + s) * pps
            st.slots[s]["left"][:] = left[a:a + pps].reshape(pps, h, w * c)
            st.slots[s]["right"][:] = right[a:a + pps].reshape(pps, h, w * c)
            st.submit(s)
        assert ctx.last_kernel in ("dense_corr_argmin_kernel", "dense_corr_mma_kernel", "dense_corr_umma_kernel")
        for s in range(n_slots):
            st.wait(s)
            a = (rnd * n_slots + s) * pps
            assert np.array_equal(st.slots[s]["out"]["right_index"], exp["right_index"][a:a + pps]), (rnd, s)
    st.close()


@pytest.mark.gpu
def test_raw_cost_u16_is_lossless_or_refused(ctx, oracle):
    """raw_cost_u16 (include/usv_b200.h): same costs as raw_cost for templates whose SAD fits 16 bits, 0xFFFF for
    windows without candidates, USV_ERR_UNSUPPORTED otherwise."""
    left, right = synth.make_pairs(2, 200, 40, 1, shift=9, noise_sigma=2.0, seed=5)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_min=3, search_max=40)
    mask = _abi.OUT_RAW_COST | _abi.OUT_RAW_COST_U16 | _abi.OUT_DISPARITY_U16
    got = ctx.match_dense(left, right, p, mask=mask)
    exp = oracle.match_dense(left, right, p, mask=mask)
    assert np.array_equal(got["raw_cost_u16"], exp["raw_cost_u16"])
    assert np.array_equal(got["raw_cost_u16"], got["raw_cost"].astype(np.uint16))
    assert (got["raw_cost_u16"][:, :3] == 0xFFFF).all()  # x < search_min: no candidate
    big = _abi.make_params(tmpl_w=32, tmpl_h=32, cost="sad", search_max=40)
    with pytest.raises(api.UsvError):
        ctx.match_dense(left, right, big, mask=_abi.OUT_RAW_COST_U16)
    ssd = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="ssd", search_max=40)
    with pytest.raises(api.UsvError):
        ctx.match_dense(left, right, ssd, mask=_abi.OUT_RAW_COST_U16)


# ---- ResolveMatchList on the GPU (usv_resolve.cu) against the restatement and the reference's own lines ----------
RESOLVE_KAT = [  # SURVEY.md section 4: produced by running P/Main.cpp:432-477 itself
    ([(0, 0, .5), (0, 1, .3), (0, 2, .4), (0, 3, .1), (0, 4, .2)], [(0, 3, .1), (0, 3, .1), (0, 4, .2)]),
    ([(0, 0, .3), (0, 1, .3), (0, 2, .5)], [(0, 0, .3), (0, 1, .3), (0, 2, .5)]),
    ([(0, 0, .5), (0, 1, .2), (1, 0, .1), (1, 1, .3)], [(0, 1, .2), (1, 0, .1), (1, 1, .3)]),
    ([(0, 0, .5), (1, 1, .6), (0, 1, .1)], [(0, 1, .1), (0, 1, .1)]),
]


def _m(rows):
    return np.array(rows, dtype=_abi.MATCH_DTYPE) if len(rows) else np.zeros(0, _abi.MATCH_DTYPE)


@pytest.mark.parametrize("inp,exp", RESOLVE_KAT)
def test_gpu_resolve_known_answers(ctx, inp, exp):
    assert ctx.resolve_match_list(_m(inp)).tobytes() == _m(exp).tobytes()
    assert ctx.last_kernel == "resolve_next_smaller_kernel"


def test_gpu_resolve_random_vs_oracle_and_reference(ctx, oracle):
    rng = np.random.default_rng(432)
    ref_ok = oracle.ref() is not None
    assert len(ctx.resolve_match_list(_m([]))) == 0
    for t in range(120):
        n = int(rng.integers(1, 400))
        k = int(rng.integers(1, 12))
        m = np.zeros(n, _abi.MATCH_DTYPE)
        m["LeftIndex"], m["RightIndex"] = rng.integers(0, k, n), rng.integers(0, k, n)
        m["MatchValue"] = rng.integers(0, 10, n) / 8.0  # many ties: the strict '>' of :451 matters
        if t % 5 == 0:
            m["MatchValue"][rng.integers(0, n, 1 + n // 6)] = np.nan
        if t % 7 == 0:
            m["MatchValue"][rng.integers(0, n, 1 + n // 6)] = np.inf
        got = ctx.resolve_match_list(m)
        assert got.tobytes() == oracle.resolve_match_list(m).tobytes(), t
        if ref_ok:
            assert got.tobytes() == oracle.ref_resolve_match_list(m).tobytes(), t


def test_gpu_resolve_long_lists(ctx, oracle):
    """One giant group (the sequential worst case of the per-group stack pass) and the dense winners of a real
    frame pair (distinct LeftIndex, conflicts through RightIndex only, NO_MATCH records skipped)."""
    rng = np.random.default_rng(7)
    n = 20000
    m = np.zeros(n, _abi.MATCH_DTYPE)
    m["LeftIndex"], m["RightIndex"] = 3, rng.integers(0, 50, n)
    m["MatchValue"] = rng.random(n)
    assert ctx.resolve_match_list(m).tobytes() == oracle.resolve_match_list(m).tobytes()
    left, right = synth.make_pairs(1, 160, 40, 1, shift=9, noise_sigma=2.0, seed=11)
    p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="sad", search_min=2, search_max=30, accept_threshold=0.05)
    win = ctx.match_dense(left, right, p, mask=_abi.OUT_MATCHES)["matches"][0]
    kept = win[win["RightIndex"] != _abi.NO_MATCH]
    assert 0 < len(kept) < len(win)
    exp = oracle.resolve_match_list(kept)
    assert ctx.resolve_match_list(win, skip_unmatched=True).tobytes() == exp.tobytes()
    assert ctx.resolve_match_list(kept).tobytes() == exp.tobytes()
    assert len(exp) <= len(kept)


def test_gpu_id_matcher_vs_oracle_and_reference(ctx, oracle):
    """IDMatcher (P/Main.cpp:483-499) on the GPU, comma-operator quirk of :492 included."""
    cur = _m([(0, 5, .1), (1, 7, .2), (2, 5, .3)])
    old = _m([(5, 9, .1), (7, 3, .2), (8, 1, .3)])
    assert ctx.id_matcher(cur, old).tolist() == [[9, 0, 0], [3, 0, 0], [9, 0, 0]]
    assert len(ctx.id_matcher(cur, _m([]))) == 0 and len(ctx.id_matcher(_m([]), old)) == 0
    rng = np.random.default_rng(483)
    ref_ok = oracle.ref() is not None
    for _ in range(40):
        a, b = np.zeros(int(rng.integers(1, 300)), _abi.MATCH_DTYPE), np.zeros(int(rng.integers(1, 300)), _abi.MATCH_DTYPE)
        for m in (a, b):
            m["LeftIndex"], m["RightIndex"] = rng.integers(0, 20, len(m)), rng.integers(0, 20, len(m))
        got = ctx.id_matcher(a, b).tolist()
        assert got == oracle.id_matcher(a, b).tolist()
        if ref_ok:
            assert got == oracle.ref_id_matcher(a, b).tolist()


def test_unsynchronised_extrapolation(ctx, oracle):
    """SURVEY 8f-2: an object that moves between the other camera's frames is ranged at THIS camera's capture time
    by tracking it through three frames and extrapolating (P/DistanceCalculator.cpp:53-84). Constant pixel velocity:
    the shift grows by 3 px per 33 ms frame; this camera fires 22 ms after the other camera's newest frame."""
    from unsynchronized_stereo_vision_proj325_b200 import pipeline
    shifts, t_other, t_this = (31, 34, 37), (0.000, 0.033, 0.066), 0.088
    frames = [synth.make_pairs(1, 320, 64, 1, shift=s, noise_sigma=0.0, seed=9) for s in shifts]
    left = frames[0][0][0]
    assert all(np.array_equal(f[0][0], left) for f in frames)  # same seed: one left frame, three right frames
    others = [f[1][0] for f in frames]
    tpl = np.array([[100, 10], [150, 20], [200, 30], [260, 40]], np.int32)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_max=60, distance_kind=_abi.DIST_POWERLAW)
    res = pipeline.extrapolated_distances(ctx, _abi.LEFT_CAM, left, t_this, others, t_other, tpl, p)
    assert res["accepted"].all()
    assert np.array_equal(res["tracks"], np.array([tpl[:, 0] - s for s in shifts], np.float32))
    # constant velocity 3 px / 33 ms -> at t_this the other camera would see the object 2 px further: disparity 39
    exp_now = oracle.distance([39], _abi.DIST_POWERLAW)[0]
    assert np.allclose(res["distance"], exp_now, rtol=1e-12)
    assert np.allclose(res["nearest_distance"], oracle.distance([37], _abi.DIST_POWERLAW)[0], rtol=1e-12)
    # and bit for bit what the restated reference function gives on the same centre points
    half = 8.0
    cen = lambda xs: np.stack([xs + half, tpl[:, 1] + half], 1).astype(np.float32)  # noqa: E731
    ns = lambda t: int(round(t * 1e9))  # noqa: E731
    exp = oracle.moving_object_distance(_abi.LEFT_CAM, ns(t_this), cen(tpl[:, 0].astype(np.float32)), cen(res["tracks"][2]),
                                        cen(res["tracks"][1]), cen(res["tracks"][0]), np.repeat(np.arange(4)[:, None], 3, 1),
                                        ns(t_other[2]), ns(t_other[1]), ns(t_other[0]))
    assert np.allclose(res["distance"], exp, rtol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("cost,n", [("sad", 100), ("zncc", 70)])
def test_many_pairs_block_order(ctx, oracle, cost, n):
    """The dense kernels run a one-dimensional grid: chunks of up to 64 pairs, inside a chunk tile-major with the heaviest
    x-tile first. More pairs than one chunk, the last chunk partly filled, several x-tiles and bands: every pair, every
    window against the oracle."""
    w, h = 150, 36
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost=cost)
    left, right = synth.make_pairs(n, w, h, 1, shift=9, noise_sigma=2.0, seed=77)
    got = ctx.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_DISPARITY_U16)
    exp = oracle.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_DISPARITY_U16)
    assert ctx.last_kernel in (("dense_sad_argmin_kernel",) if cost == "sad" else ("dense_corr_mma_kernel", "dense_corr_umma_kernel"))
    for k in ("right_index", "disparity_u16"):
        assert np.array_equal(got[k], exp[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("lo,n_disp", [(0, 32), (0, 64), (0, 128), (0, 256), (4, 128), (5, 128), (-8, 64), (0, 125), (0, 29), (0, 1), (3, 4)])
def test_bounded_ranges_thin_last_pass(ctx, oracle, side, lo, n_disp):
    """Ranges whose length is a multiple of 32 (or up to 3 short of one) end in the thin pass of the SAD kernel (one
    disparity per thread for the last 1..3 disparities of three of the four byte phases); neighbours of those lengths
    and offsets that are not multiples of 4 take the regular path. Both camera sides, frames wide enough for interior
    tiles (all runs equal) and edge tiles (range clipped by the frame)."""
    w, h = 420, 30
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_min=lo, search_max=lo + n_disp - 1, camera_side=side)
    left, right = synth.make_pairs(2, w, h, 1, shift=21 if side == 0 else -21, noise_sigma=2.0, seed=5 + n_disp)
    got = ctx.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST)
    exp = oracle.match_dense(left, right, p, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST)
    assert ctx.last_kernel == "dense_sad_argmin_kernel"
    for k in ("right_index", "raw_cost"):
        assert np.array_equal(got[k], exp[k]), k


def _resolved_map_from_reference(oracle, got_pair, nx, use_ref):
    """The reference's ResolveMatchList (restated, or its own lines compiled verbatim) over the accepted winners of one
    pair -> the disparity map in which only the windows whose record is in TentativeMatch keep their disparity."""
    win = got_pair["matches"]
    kept = win[win["RightIndex"] != _abi.NO_MATCH]
    out = (oracle.ref_resolve_match_list if use_ref else oracle.resolve_match_list)(kept)
    alive = np.zeros(len(win), bool)
    alive[np.unique(out["LeftIndex"])] = True
    # every output record is one of the winners, unchanged
    assert all(win[int(m["LeftIndex"])].tobytes() == m.tobytes() for m in out[:: max(1, len(out) // 200)])
    return np.where(alive, got_pair["disparity_u16"], _abi.NO_DISPARITY).astype(np.uint16)


RESOLVED_MAP_CASES = [
    ("sad", _abi.LEFT_CAM, 200, 40, 16, 16, dict()),
    ("sad", _abi.RIGHT_CAM, 131, 30, 8, 8, dict(search_max=40)),
    ("ssd", _abi.LEFT_CAM, 150, 28, 12, 12, dict(search_min=2, search_max=60, accept_threshold=0.05)),
    ("zncc", _abi.LEFT_CAM, 160, 30, 16, 16, dict(search_max=63)),
    ("ncc", _abi.RIGHT_CAM, 140, 26, 9, 7, dict(search_max=50, accept_threshold=0.3)),
    ("sad", _abi.LEFT_CAM, 96, 24, 11, 4, dict(stride_x=2, stride_y=3, search_max=40)),   # direct-form kernel
    ("sad", _abi.LEFT_CAM, 120, 26, 8, 8, dict(search_min=-12, search_max=30)),           # negative disparities: resolved from RightIndex
    ("ssd", _abi.RIGHT_CAM, 120, 26, 8, 8, dict(search_min=-20, search_max=25)),
]


def resolved_map_inputs(cost, side, w, h, tw, th, kw):
    """Frames with flat and repeated regions, so that many windows claim the same RightIndex with equal and with
    different values. Also rebuilt by tests/golden/make_ref_answers.py."""
    left, right = synth.make_pairs(2, w, h, 1, shift=9 if side == _abi.LEFT_CAM else -9, noise_sigma=2.0, seed=w + h)
    left[0, :, w // 2:] = 77                      # flat half: all-tie rows of candidates
    right[0, :, : w // 3] = right[0, :, w // 3: 2 * (w // 3)]  # repeated texture: two windows, one best x'
    right[1] = np.roll(right[1], 1, axis=0) // 2
    return left, right, _abi.make_params(tmpl_w=tw, tmpl_h=th, cost=cost, camera_side=side, **kw)


@pytest.mark.parametrize("cost,side,w,h,tw,th,kw", RESOLVED_MAP_CASES)
def test_resolved_disparity_map(ctx, oracle, cost, side, w, h, tw, th, kw):
    """usv_outputs.resolved_disparity_u16: ResolveMatchList (P/Main.cpp:432-477) over the dense winners on the device."""
    left, right, p = resolved_map_inputs(cost, side, w, h, tw, th, kw)
    full = api.ALL_OUTPUTS | _abi.OUT_RESOLVED_DISPARITY_U16
    got = ctx.match_dense(left, right, p, mask=full)
    f = _abi.frame_desc_for(left)
    nx, ny, _ = api.grid_dims(f, p)
    n_beaten = 0
    for pair in range(2):
        gp = {k: v[pair] for k, v in got.items()}
        exp = _resolved_map_from_reference(oracle, gp, nx, use_ref=(pair == 0))
        assert np.array_equal(gp["resolved_disparity_u16"], exp)
        n_beaten += int(((exp == _abi.NO_DISPARITY) & (gp["disparity_u16"] != _abi.NO_DISPARITY)).sum())
    assert n_beaten > 0  # the case exercises the conflict rule
    # the same map when the winners come from right_index + raw_cost, and from the library's own scratch
    for mask in (_abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST | _abi.OUT_RESOLVED_DISPARITY_U16, _abi.OUT_RESOLVED_DISPARITY_U16):
        again = ctx.match_dense(left, right, p, mask=mask)
        assert np.array_equal(again["resolved_disparity_u16"], got["resolved_disparity_u16"])


def test_distance_lut_matches_epilogue(ctx, oracle):
    for kind in (_abi.DIST_PINHOLE, _abi.DIST_POWERLAW):
        lut = ctx.distance_lut(kind, 700)
        exp = oracle.distance(np.arange(700), kind)
        assert np.array_equal(np.isinf(lut), np.isinf(exp))
        fin = np.isfinite(exp)
        assert np.allclose(lut[fin], exp[fin], rtol=DIST_RTOL, atol=0)
    left, right = synth.make_pairs(1, 128, 24, 1, shift=7, noise_sigma=1.0, seed=3)
    got = ctx.match_dense(left, right, _abi.make_params(tmpl_w=8, tmpl_h=8, cost="sad"))
    d = got["disparity_u16"][0]
    ok = d != _abi.NO_DISPARITY
    assert np.array_equal(got["distance"][0][ok], ctx.distance_lut(_abi.DIST_PINHOLE, 128)[d[ok]])  # same table, bit for bit


BLOCK_SEARCH_COSTS = ["sad", "zncc"]


def block_search_inputs(cost):
    """Also rebuilt by tests/golden/make_ref_answers.py."""
    left, right = synth.make_pairs(1, 150, 36, 1, shift=9, noise_sigma=2.0, seed=5)
    left[0, :, 100:] = 60  # a flat region: many windows claim the same candidate
    return left, right, _abi.make_params(tmpl_w=12, tmpl_h=12, cost=cost, search_max=60, distance_kind=_abi.DIST_POWERLAW)


@pytest.mark.parametrize("cost", BLOCK_SEARCH_COSTS)
def test_block_search_host_is_generate_resolve_distance(ctx, oracle, cost):
    """usv_block_search_host = the reference's call order (P/Main.cpp:1115-1143, :681-694) in one call: equal, entry for entry,
    to the reference's own ResolveMatchList (compiled verbatim) over the oracle's accepted winners, with each entry's distance."""
    left, right, p = block_search_inputs(cost)
    got_m, got_d = ctx.block_search(left[0], right[0], p)
    exp = oracle.match_dense(left, right, p)
    win = exp["matches"][0]
    kept = win[win["RightIndex"] != _abi.NO_MATCH]
    exp_list = oracle.ref_resolve_match_list(kept)
    assert got_m.tobytes() == exp_list.tobytes()
    exp_d = exp["distance"][0][exp_list["LeftIndex"]]
    assert np.array_equal(np.isinf(got_d), np.isinf(exp_d))
    fin = np.isfinite(exp_d)
    assert np.allclose(got_d[fin], exp_d[fin], rtol=DIST_RTOL, atol=0)
    assert len(got_m) < len(kept) or len(np.unique(kept["RightIndex"])) == len(kept)


def test_stream_submit_io_lands_in_caller_arrays(ctx, oracle):
    """usv_stream_submit_io: frames from and results into caller-owned (page-locked) arrays, disjoint slices per submission."""
    left, right = synth.make_pairs(6, 160, 40, 1, shift=11, noise_sigma=2.0, seed=8)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_max=63)
    f = _abi.frame_desc_for(left)
    nx, ny, _ = api.grid_dims(f, p)
    mask = _abi.OUT_RESOLVED_DISPARITY_U16 | _abi.OUT_RAW_COST_U16
    res = np.zeros((6, nx * ny), np.uint16)
    cost = np.zeros((6, nx * ny), np.uint16)
    for a in (left, right, res, cost):
        ctx.host_register(a)
    st = ctx.stream(f, p, pairs_per_slot=2, n_slots=2, mask=mask)
    try:
        for k in range(3):
            slot = k % 2
            if k >= 2:
                st.wait(slot)
            st.submit_io(slot, left[2 * k:2 * k + 2], right[2 * k:2 * k + 2],
                         {"resolved_disparity_u16": res[2 * k:2 * k + 2], "raw_cost_u16": cost[2 * k:2 * k + 2]})
        st.wait(0)
        st.wait(1)
    finally:
        st.close()
        for a in (left, right, res, cost):
            ctx.host_unregister(a)
    ref = ctx.match_dense(left, right, p, mask=mask)
    assert np.array_equal(res, ref["resolved_disparity_u16"]) and np.array_equal(cost, ref["raw_cost_u16"])
    exp = oracle.match_dense(left, right, p, mask=_abi.OUT_RAW_COST)
    assert np.array_equal(cost.astype(np.uint32), exp["raw_cost"])


def test_device_api_out_of_frame_template_is_no_match(ctx, oracle):
    """ADVICE r1: a template list in HBM cannot be validated by the host; a template that does not fit the frame gets the
    "no candidate" record instead of an out-of-bounds strip, and its neighbours in the list are unaffected."""
    torch = pytest.importorskip("torch")
    left, right = synth.make_pairs(1, 128, 32, 1, shift=7, noise_sigma=2.0, seed=4)
    dl, dr = torch.from_numpy(np.ascontiguousarray(left)).cuda(), torch.from_numpy(np.ascontiguousarray(right)).cuda()
    f = _abi.frame_desc_for(left)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad")
    tx = torch.tensor([40, 113, -1, 60, 5000], dtype=torch.int32).cuda()   # 113 = nxc: one past the last valid x
    ty = torch.tensor([3, 3, 3, 17, 3], dtype=torch.int32).cuda()          # 17 = nyc: one past the last valid y
    o_ri = torch.zeros(5, dtype=torch.int32).cuda()
    o_rc = torch.zeros(5, dtype=torch.int32).cuda()
    out = _abi.Outputs()
    out.right_index, out.raw_cost = o_ri.data_ptr(), o_rc.data_ptr()
    ctx.match_templates_device(dl.data_ptr(), dr.data_ptr(), f, 1, tx.data_ptr(), ty.data_ptr(), 5, p, out, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ri = o_ri.cpu().numpy().view(np.uint32)
    exp = oracle.match_templates(left, right, [40], [3], p, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST)
    assert ri[0] == exp["right_index"][0, 0] and o_rc.cpu().numpy().view(np.uint32)[0] == exp["raw_cost"][0, 0]
    assert (ri[1:] == _abi.NO_MATCH).all()
    assert api.lib().usv_device_status(ctx._h) == 0


def test_destroy_refuses_while_a_stream_is_open():
    """ADVICE r1: usv_destroy with a live usv_stream would leave the stream with a dangling context; it is refused instead,
    and the Python Context closes its streams first."""
    import ctypes as C
    L = api.lib()
    h = C.c_void_p()
    assert L.usv_create(0, C.byref(h)) == 0
    f = _abi.FrameDesc(64, 32, 1, 64, 64 * 32)
    p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="sad")
    s = C.c_void_p()
    assert L.usv_stream_create(h, C.byref(f), C.byref(p), C.c_int32(2), C.c_int32(2), C.c_uint32(_abi.OUT_DISPARITY_U16), C.byref(s)) == 0
    assert L.usv_destroy(h) == _abi.USV_ERR_INVALID_ARG
    assert b"usv_stream" in L.usv_last_error(h)
    L.usv_stream_destroy.argtypes = [C.c_void_p]
    assert L.usv_stream_destroy(s) == 0
    assert L.usv_destroy(h) == 0
    c = api.Context(0)
    st = c.stream(f, p, pairs_per_slot=2, n_slots=2, mask=_abi.OUT_DISPARITY_U16)
    c.close()            # closes the stream first
    assert st._h is None


@pytest.mark.parametrize("cost,kw", [
    ("sad", dict(search_max=60)),
    ("sad", dict(search_min=-9, search_max=40)),            # negative disparities: the resolve reads RightIndex
    ("ssd", dict(search_min=-5, search_max=50, accept_threshold=0.05)),
    ("zncc", dict(search_min=-6, search_max=40)),
    ("sad", dict(search_max=40, stride_x=2, stride_y=2)),   # direct-form kernel
])
def test_every_output_subset_gives_the_same_arrays(ctx, oracle, cost, kw):
    """The library serves any subset of usv_outputs; arrays it needs itself (the winners the row resolve reads) come from the caller's
    set or from scratch, depending on the subset. Every subset must reproduce the arrays of the full set, bit for bit."""
    left, right = synth.make_pairs(2, 150, 30, 1, shift=8, noise_sigma=2.0, seed=77)
    left[1, :, 70:] = 50
    p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost=cost, **kw)
    u16 = _abi.OUT_RAW_COST_U16 if cost == "sad" else 0  # the 16-bit cost exists for SAD only
    full_mask = api.ALL_OUTPUTS | u16 | _abi.OUT_RESOLVED_DISPARITY_U16
    full = ctx.match_dense(left, right, p, mask=full_mask)
    exp = oracle.match_dense(left, right, p)
    for k in ("right_index", "raw_cost", "disparity_u16"):
        assert np.array_equal(full[k], exp[k]), k
    rng = np.random.default_rng(11)
    bits = [_abi.OUT_MATCHES, _abi.OUT_RIGHT_INDEX, _abi.OUT_RAW_COST, _abi.OUT_SCORE, _abi.OUT_DISTANCE, _abi.OUT_DISTANCE_F32,
            _abi.OUT_DISPARITY_U16] + ([u16] if u16 else [])
    masks = [_abi.OUT_RESOLVED_DISPARITY_U16 | b for b in [0] + bits]
    masks += [_abi.OUT_RESOLVED_DISPARITY_U16 | _abi.OUT_DISPARITY_U16 | u16,
              _abi.OUT_RESOLVED_DISPARITY_U16 | _abi.OUT_DISPARITY_U16 | _abi.OUT_RAW_COST,
              _abi.OUT_RESOLVED_DISPARITY_U16 | _abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST,
              _abi.OUT_RESOLVED_DISPARITY_U16 | _abi.OUT_RIGHT_INDEX | u16]
    masks += [int(sum(b for b in bits if rng.random() < 0.4)) | (_abi.OUT_RESOLVED_DISPARITY_U16 if rng.random() < 0.7 else 0) for _ in range(16)]
    for m in masks:
        if m == 0:
            continue
        got = ctx.match_dense(left, right, p, mask=m)
        for k, v in got.items():
            assert v.tobytes() == full[k].tobytes(), (hex(m), k)
