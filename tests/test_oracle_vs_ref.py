"""Pin the oracle against the reference's own code compiled verbatim
(oracle/_ref: P/Match.cpp, P/DistanceCalculator.cpp, P/Main.cpp:432-477), or against
that code's answers recorded in tests/golden/ref_answers.npz when it is not built, and
against the known answers recorded from it in SURVEY.md section 4."""
import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi

M = _abi.MATCH_DTYPE


def _m(lst):
    return np.array(lst, dtype=M)


RESOLVE_KAT = [
    ([(0, 0, .5), (0, 1, .3), (0, 2, .4), (0, 3, .1), (0, 4, .2)], [(0, 3, .1), (0, 3, .1), (0, 4, .2)]),
    ([(0, 0, .3), (0, 1, .3), (0, 2, .5)], [(0, 0, .3), (0, 1, .3), (0, 2, .5)]),
    ([(0, 0, .5), (0, 1, .2), (1, 0, .1), (1, 1, .3)], [(0, 1, .2), (1, 0, .1), (1, 1, .3)]),
    ([(0, 0, .5), (1, 1, .6), (0, 1, .1)], [(0, 1, .1), (0, 1, .1)]),
    ([], []),
]


@pytest.mark.parametrize("inp,exp", RESOLVE_KAT)
def test_resolve_known_answers(oracle, inp, exp):
    got = oracle.resolve_match_list(_m(inp))
    assert got.tolist() == _m(exp).tolist()


@pytest.mark.parametrize("inp,exp", RESOLVE_KAT)
def test_ref_resolve_known_answers(oracle, inp, exp):
    got = oracle.ref_resolve_match_list(_m(inp))
    assert got.tolist() == _m(exp).tolist()


def test_resolve_random_vs_ref(oracle):
    rng = np.random.default_rng(325)
    for trial in range(200):
        n = int(rng.integers(0, 40))
        m = np.zeros(n, dtype=M)
        m["LeftIndex"] = rng.integers(0, 6, n)
        m["RightIndex"] = rng.integers(0, 6, n)
        # coarse values so that exact ties occur
        m["MatchValue"] = rng.integers(0, 8, n) / 8.0
        a = oracle.resolve_match_list(m)
        b = oracle.ref_resolve_match_list(m)
        assert a.tobytes() == b.tobytes(), trial


def test_single_template_resolve_is_first_min(oracle):
    """ResolveMatchList fed one template's candidates: out[0] is the first
    minimum in scan order (strict '>' at P/Main.cpp:451)."""
    rng = np.random.default_rng(1)
    for _ in range(100):
        n = int(rng.integers(1, 50))
        v = rng.integers(0, 6, n) / 8.0
        m = np.zeros(n, dtype=M)
        m["RightIndex"] = np.arange(n)
        m["MatchValue"] = v
        out = oracle.ref_resolve_match_list(m)
        assert out[0]["RightIndex"] == int(np.argmin(v))  # np.argmin = first minimum
        assert out[0]["MatchValue"] == v.min()


def test_match_layout(oracle):
    assert oracle.ref_sizeof_match() == 16 == M.itemsize
    assert (M.fields["LeftIndex"][1], M.fields["RightIndex"][1], M.fields["MatchValue"][1]) == (0, 4, 8)


def test_distance_known_answers(oracle):
    # SURVEY section 4: power law / pinhole at several disparities (reference arithmetic)
    kat = {1: (35380.1758, 18753.4884), 8: (3405.5690, 2344.1860), 16: (1560.7485, 1172.0930),
           64: (327.8079, 293.0233), 128: (150.2321, 146.5116), 256: (68.8503, 73.2558)}
    for d, (pl, ph) in kat.items():
        assert oracle.distance([d], _abi.DIST_POWERLAW)[0] == pytest.approx(pl, rel=1e-6)
        assert oracle.distance([d], _abi.DIST_PINHOLE)[0] == pytest.approx(ph, rel=1e-6)
    assert oracle.distance([40], _abi.DIST_POWERLAW)[0] == pytest.approx(556.401951467, rel=1e-11)
    assert np.isinf(oracle.distance([0], _abi.DIST_POWERLAW)[0])
    assert np.isinf(oracle.distance([0], _abi.DIST_PINHOLE)[0])


MS = 1_000_000


def _moving_case():
    # other camera x = 240, 250, 260 at t = 33, 67, 100 ms; this x = 300 at 110 ms (SURVEY section 4)
    return dict(t_this=110 * MS, this_xy=[(300, 200)], other_xy=[(260, 200)], old_xy=[(250, 200)],
                older_xy=[(240, 200)], idx3=[(0, 0, 0)], t_other=100 * MS, t_old=67 * MS, t_older=33 * MS)


def _call(fn, side, c):
    return fn(side, c["t_this"], c["this_xy"], c["other_xy"], c["old_xy"], c["older_xy"], c["idx3"],
              c["t_other"], c["t_old"], c["t_older"])


def test_moving_known_answer(oracle):
    c = _moving_case()
    a = _call(oracle.moving_object_distance, 1, c)
    b = _call(oracle.ref_moving_object_distance, 1, c)
    assert b[0] == pytest.approx(626.463714398, rel=1e-11)
    assert a.tobytes() == b.tobytes()


def test_moving_random_vs_ref(oracle):
    rng = np.random.default_rng(7)
    for trial in range(300):
        n_other, n_old, n_older = (int(rng.integers(0 if trial % 10 == 0 else 1, 6)) for _ in range(3))
        n_idx, n_this = int(rng.integers(0, 8)), int(rng.integers(0, 8))
        c = dict(
            this_xy=rng.uniform(0, 640, (n_this, 2)), other_xy=rng.uniform(0, 640, (n_other, 2)),
            old_xy=rng.uniform(0, 640, (n_old, 2)), older_xy=rng.uniform(0, 640, (n_older, 2)),
            idx3=rng.integers(-1, 7, (n_idx, 3)),  # out-of-range and negative indices included
            t_older=int(rng.integers(0, 10**9)),
        )
        c["t_old"] = c["t_older"] + int(rng.integers(1, 50 * MS))
        c["t_other"] = c["t_old"] + int(rng.integers(1, 50 * MS))
        c["t_this"] = c["t_other"] + int(rng.integers(-20 * MS, 20 * MS))
        for side in (0, 1):
            a = _call(oracle.moving_object_distance, side, c)
            b = _call(oracle.ref_moving_object_distance, side, c)
            assert a.tobytes() == b.tobytes(), (trial, side)


def test_coordinates_known_answers(oracle):
    for side, exp in ((1, (9.103702, 99.584751, 12.454575)), (0, (-18.505677, 98.272783, 8.532612))):
        a = oracle.coordinate_position(side, [100.0], [(300, 200)])
        b = oracle.ref_coordinate_position(side, [100.0], [(300, 200)])
        assert a[0] == pytest.approx(exp, abs=1e-6)
        assert a.tobytes() == b.tobytes()


def test_coordinates_random_vs_ref(oracle):
    rng = np.random.default_rng(3)
    dist = rng.uniform(15, 2000, 500)
    xy = np.stack([rng.uniform(0, 640, 500), rng.uniform(0, 480, 500)], 1)
    for side in (0, 1):
        a = oracle.coordinate_position(side, dist, xy)
        b = oracle.ref_coordinate_position(side, dist, xy)
        assert a.tobytes() == b.tobytes()  # NaNs included, bit for bit


def test_deg_rad(oracle):
    for v in (0.0, 1.0, 45.0, 70.0, 180.0, -33.3):
        assert oracle.lib().usv_oracle_deg2rad(v) == oracle.ref_deg2rad(v)
        assert oracle.lib().usv_oracle_rad2deg(v) == oracle.ref_rad2deg(v)


def test_id_matcher_vs_ref(oracle):
    """IDMatcher (P/Main.cpp:483-499) incl. the comma-operator quirk at :492: triples are (old.Right, 0, 0)."""
    cur = _m([(0, 5, .1), (1, 7, .2), (2, 5, .3)])
    old = _m([(5, 9, .1), (7, 3, .2), (8, 1, .3)])
    assert oracle.ref_id_matcher(cur, old).tolist() == [[9, 0, 0], [3, 0, 0], [9, 0, 0]]
    rng = np.random.default_rng(4)
    for _ in range(100):
        a = np.zeros(int(rng.integers(0, 12)), dtype=M)
        b = np.zeros(int(rng.integers(0, 12)), dtype=M)
        for z in (a, b):
            z["LeftIndex"] = rng.integers(0, 6, len(z))
            z["RightIndex"] = rng.integers(0, 6, len(z))
        assert oracle.id_matcher(a, b).tolist() == oracle.ref_id_matcher(a, b).tolist()
