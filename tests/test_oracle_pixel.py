"""CPU: the pixel-cost oracle against the committed golden fixtures, an
independent numpy restatement, and cv2.matchTemplate (argmin / NCC cross-check;
cv2 4.13 is float32/DFT, so values are compared with a tolerance, indices exactly)."""
import glob
import os

import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, synth

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _golden_cases():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.CASES


CASES = _golden_cases()


def test_golden_files_present():
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
    # tests/test_contours.py, tests/test_preprocess_oracle.py, the reference's answers (oracle.ref_*)
    other = ("contours_cv2", "preprocess_cv2", "ref_answers")
    assert [n for n in names if n not in other] == sorted(CASES)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_golden(oracle, name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    p = _abi.make_params(**CASES[name][5])
    out = oracle.match_dense(z["left"], z["right"], p)
    for k, v in out.items():
        assert v.tobytes() == z["out_" + k].tobytes(), k


def _numpy_costs(left, right, x, y, tw, th, kind):
    """all candidate costs of template (x, y) for x' = 0..W-tw, float64/int64 numpy"""
    t = left[y:y + th, x:x + tw].astype(np.int64)
    W = left.shape[1]
    out = []
    for xr in range(W - tw + 1):
        c = right[y:y + th, xr:xr + tw].astype(np.int64)
        if kind == "sad":
            out.append(np.abs(t - c).sum())
        elif kind == "ssd":
            out.append(((t - c) ** 2).sum())
        else:
            n = t.size
            sab, sa, sb, saa, sbb = (t * c).sum(), t.sum(), c.sum(), (t * t).sum(), (c * c).sum()
            if kind == "ncc":
                out.append(0.0 if saa == 0 or sbb == 0 else float(sab) * (1.0 / np.sqrt(float(saa))) * (1.0 / np.sqrt(float(sbb))))
            else:
                num, da, db = n * sab - sa * sb, n * saa - sa * sa, n * sbb - sb * sb
                out.append(0.0 if da == 0 or db == 0 else float(num) * (1.0 / np.sqrt(float(da))) * (1.0 / np.sqrt(float(db))))
    return np.array(out)


@pytest.mark.parametrize("kind", ["sad", "ssd", "ncc", "zncc"])
def test_oracle_rows_vs_numpy(oracle, kind):
    left, right = synth.make_pairs(1, 64, 24, 1, shift=9, noise_sigma=2.0, seed=5)
    p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost=kind, search_min=-(1 << 20), search_max=1 << 20)  # every x'
    tx, ty = [0, 20, 56], [0, 7, 16]
    out = oracle.match_templates(left, right, tx, ty, p, rows=True)
    for i, (x, y) in enumerate(zip(tx, ty)):
        ref = _numpy_costs(left[0], right[0], x, y, 8, 8, kind)
        if kind in ("sad", "ssd"):
            assert out["cost_rows"][0, i, :len(ref)].tolist() == ref.tolist()
            assert out["raw_cost"][0, i] == ref.min()
            assert out["right_index"][0, i] == y * 57 + int(np.argmin(ref))
        else:
            np.testing.assert_array_equal(out["score_rows"][0, i, :len(ref)], ref)
            j = int(np.argmin(1.0 - ref))
            assert out["score"][0, i] == ref[j]


def test_tie_breaking_first_minimum(oracle):
    """Flat frames: every candidate costs 0 -> the first in scan order (smallest x') wins (P/Main.cpp:451)."""
    left = np.full((1, 20, 48), 77, np.uint8)
    right = left.copy()
    for side in (_abi.LEFT_CAM, _abi.RIGHT_CAM):
        p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="sad", camera_side=side, search_max=12)
        out = oracle.match_dense(left, right, p)
        nx = 41
        for x in (0, 5, 20, 40):
            ri = out["right_index"][0, 3 * nx + x]
            exp_x = max(0, x - 12) if side == _abi.LEFT_CAM else x
            assert ri == 3 * nx + exp_x
            assert out["raw_cost"][0, 3 * nx + x] == 0


def test_known_shift_recovered(oracle):
    left, right = synth.make_pairs(1, 128, 32, 1, shift=21, seed=9)
    p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad")
    out = oracle.match_dense(left, right, p)
    nx = 113
    d = out["disparity_u16"][0].reshape(17, nx)
    assert (d[:, 21:] == 21).all()  # windows whose true match is inside the frame
    assert (out["raw_cost"][0].reshape(17, nx)[:, 21:] == 0).all()
    dist = out["distance"][0].reshape(17, nx)[:, 21:]
    assert np.allclose(dist, ((201.6 * 4) / (21 * 0.000043)) / 1000)


def test_cv2_cross_check(oracle):
    cv2 = pytest.importorskip("cv2")
    left, right = synth.make_pairs(1, 160, 48, 1, shift=17, noise_sigma=3.0, seed=11)
    L, R = np.ascontiguousarray(left[0]), np.ascontiguousarray(right[0])
    tx, ty = [40, 90, 143], [3, 20, 31]
    every = dict(search_min=-(1 << 20), search_max=1 << 20)
    for kind, method in (("ssd", cv2.TM_SQDIFF), ("ncc", cv2.TM_CCORR_NORMED), ("zncc", cv2.TM_CCOEFF_NORMED)):
        out = oracle.match_templates(left, right, tx, ty, _abi.make_params(tmpl_w=16, tmpl_h=16, cost=kind, **every), rows=True)
        for i, (x, y) in enumerate(zip(tx, ty)):
            res = cv2.matchTemplate(R[y:y + 16], np.ascontiguousarray(L[y:y + 16, x:x + 16]), method)[0]
            if kind == "ssd":
                mine = out["cost_rows"][0, i, :len(res)].astype(np.float64)
                assert int(np.argmin(res)) == int(np.argmin(mine))
                assert np.abs(res - mine).max() <= 64  # float32 DFT error (SURVEY 8c)
            else:
                mine = out["score_rows"][0, i, :len(res)]
                assert int(np.argmax(res)) == int(np.argmax(mine))
                assert np.abs(res - mine).max() <= 1e-4


def test_sad_against_cv2_norm_l1(oracle):
    """cv2.matchTemplate has no SAD mode, so the headline cost gets its own third-party check: every candidate's cost of
    a set of templates (gray and colour, odd sizes, frame edges) against cv2.norm(a, b, NORM_L1) of the two patches — an
    implementation that shares nothing with the oracle's loops — and the winner against the first minimum of that row."""
    cv2 = pytest.importorskip("cv2")
    every = dict(search_min=-(1 << 20), search_max=1 << 20)
    for c, tw, th, w, h in ((1, 16, 16, 160, 48), (3, 32, 32, 150, 40), (1, 7, 5, 61, 19), (3, 9, 4, 40, 12)):
        left, right = synth.make_pairs(1, w, h, c, shift=11, noise_sigma=3.0, seed=70 + tw)
        L, R = np.ascontiguousarray(left[0]), np.ascontiguousarray(right[0])
        nxc, nyc = w - tw + 1, h - th + 1
        tx, ty = [0, nxc - 1, nxc // 2, 11, 12], [0, nyc - 1, nyc // 2, 1, nyc - 1]
        out = oracle.match_templates(left, right, tx, ty, _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="sad", accept_threshold=2.0, **every), rows=True)
        for i, (x, y) in enumerate(zip(tx, ty)):
            a = np.ascontiguousarray(L[y:y + th, x:x + tw])
            ref = np.array([cv2.norm(a, np.ascontiguousarray(R[y:y + th, xr:xr + tw]), cv2.NORM_L1) for xr in range(nxc)])
            assert np.array_equal(out["cost_rows"][0, i, :nxc].astype(np.float64), ref)
            assert out["raw_cost"][0, i] == ref.min() and out["right_index"][0, i] == y * nxc + int(np.argmin(ref))


def test_empty_candidate_range(oracle):
    left, right = synth.make_pairs(1, 40, 16, 1, shift=3, seed=2)
    p = _abi.make_params(tmpl_w=8, tmpl_h=8, cost="sad", search_min=10, search_max=12)
    out = oracle.match_dense(left, right, p)
    nx = 33
    assert (out["right_index"][0].reshape(9, nx)[:, :10] == _abi.NO_MATCH).all()  # x - 10 < 0: no candidates
    assert (out["raw_cost"][0].reshape(9, nx)[:, :10] == 0xFFFFFFFF).all()
    assert np.isinf(out["matches"]["MatchValue"][0].reshape(9, nx)[:, :10]).all()


@pytest.mark.parametrize("w,h,tw,th,kw", [
    (160, 40, 16, 16, dict()),                                                     # fast path, full range
    (200, 36, 16, 16, dict(search_min=3, search_max=70)),
    (131, 30, 16, 12, dict(camera_side=_abi.RIGHT_CAM, search_max=40)),
    (120, 28, 16, 16, dict(search_min=-9, search_max=9)),                          # signed range
    (97, 25, 7, 5, dict(search_max=33)),                                           # generic path
    (90, 40, 32, 32, dict(camera_side=_abi.RIGHT_CAM)),
])
def test_sliding_cpu_arm_equals_direct_form(oracle, w, h, tw, th, kw):
    """bench.py's algorithm-matched CPU arm (oracle/sliding_sad_cpu.c: column sums slid down the rows, window sums along x — the
    GPU kernel's formulation) returns exactly the direct-form oracle's winners and costs, ties included."""
    left, right = synth.make_pairs(2, w, h, 1, shift=7, noise_sigma=2.0, seed=w)
    left[1, : h // 2] = 50; right[1, : h // 2] = 50  # flat half: every candidate ties
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, cost="sad", accept_threshold=10.0, **kw)
    exp = oracle.match_dense(left, right, p)
    ri, rc, ev = oracle.match_dense_sliding(left, right, p, threads=3)
    assert np.array_equal(ri, exp["right_index"]) and np.array_equal(rc, exp["raw_cost"])
    f = _abi.frame_desc_for(left)
    assert ev == 2 * oracle.grid_dims(f, p)[2]
    # a row range only (what the bench samples)
    nx, ny, _ = oracle.grid_dims(f, p)
    ri2, rc2, _ = oracle.match_dense_sliding(left, right, p, 2, min(ny, 9))
    assert np.array_equal(ri2.reshape(2, ny, nx)[:, 2:9], exp["right_index"].reshape(2, ny, nx)[:, 2:9])
    assert np.array_equal(rc2.reshape(2, ny, nx)[:, 2:9], exp["raw_cost"].reshape(2, ny, nx)[:, 2:9])
