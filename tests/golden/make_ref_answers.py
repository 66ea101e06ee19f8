"""Records tests/golden/ref_answers.npz: the answers of the reference's own ResolveMatchList, IDMatcher and
DistanceCalculator.cpp functions (P/Main.cpp:432-499, P/Match.cpp, P/DistanceCalculator.cpp) on every input the
tests give them (`python tests/golden/make_ref_answers.py`).

The tests call that code through oracle.ref_*: compiled verbatim into oracle/_ref when the reference source is at
hand, otherwise answered from this file, keyed by a digest of each call's inputs. With oracle/_ref built this script
records from the reference itself. Without it, it records the oracle's restatement of those functions (oracle/*.c),
which is what the tests had compared with the reference's own code, byte for byte, on these same inputs while it
was built. Resolve answers are stored as positions in the input list (every output record is an input record)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle  # noqa: E402
from unsynchronized_stereo_vision_proj325_b200 import _abi  # noqa: E402

REF = oracle.ref()  # the reference's own code, or None


def _positions(m, out):
    first = {}
    for i in range(len(m)):
        first.setdefault(m[i:i + 1].tobytes(), i)
    return np.array([first[out[j:j + 1].tobytes()] for j in range(len(out))], np.uint16)


def _answer(name, inputs):
    if name == "resolve_match_list":
        (m,) = inputs
        assert len(m) < 1 << 16
        return _positions(m, oracle._resolve(REF.ref_resolve_match_list, m) if REF else oracle.resolve_match_list(m))
    if name == "id_matcher":
        return oracle._id_matcher(REF.ref_id_matcher if REF else oracle.lib().usv_oracle_id_matcher, *inputs)
    if name == "moving_object_distance":
        (side, t_this, t_other, t_old, t_older), this_xy, other_xy, old_xy, older_xy, idx3 = inputs
        fn = REF.ref_moving_object_distance if REF else oracle.lib().usv_oracle_moving_object_distance
        return oracle._moving(fn, REF is not None, side, t_this, this_xy, other_xy, old_xy, older_xy, idx3, t_other, t_old, t_older)
    if name == "coordinate_position":
        side, dist, xy = inputs
        if REF is None:
            return oracle.coordinate_position(int(side), dist, xy)
        out = np.zeros((len(dist), 3), np.float64)
        n = REF.ref_coordinate_position(int(side), oracle._ptr(dist), oracle._ptr(xy), len(dist), oracle._ptr(out))
        return out[:n]
    if name == "sizeof_match":
        return np.array([REF.ref_sizeof_match() if REF else 16], np.int32)  # P/Match.hpp: two unsigned ints and a double
    if name in ("deg2rad", "rad2deg"):
        (v,) = inputs
        fn = getattr(REF, "ref_" + name) if REF else getattr(oracle.lib(), "usv_oracle_" + name)
        return np.array([fn(float(v))], np.float64)
    raise KeyError(name)


def main():
    import pytest
    import test_gpu_parity as gp

    answers = {}

    def record(name, *inputs):
        key = (name, oracle.answer_key(name, *inputs))
        if key not in answers:
            answers[key] = _answer(name, inputs)
        return answers[key]

    oracle.ref = lambda: None  # every ref_* call goes through record()
    oracle.recorded_answer = record
    # tests/test_oracle_vs_ref.py, run as it is
    rc = pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_oracle_vs_ref.py")])
    assert rc == 0, rc
    # the GPU tests: the reference over the oracle's accepted winners of the same frames (the device's winners are
    # the oracle's, bit for bit; the resolved-map test resolves pair 0 with the reference)
    inputs = [gp.resolved_map_inputs(*case) for case in gp.RESOLVED_MAP_CASES]
    inputs += [gp.block_search_inputs(cost) for cost in gp.BLOCK_SEARCH_COSTS]
    for left, right, p in inputs:
        win = oracle.match_dense(left, right, p)["matches"][0]
        oracle.ref_resolve_match_list(win[win["RightIndex"] != _abi.NO_MATCH])
    packed = {}
    for fn in sorted({name for name, _ in answers}):
        keys = [k for name, k in answers if name == fn]
        rows = [answers[fn, k] for k in keys]
        packed[fn + ".keys"] = np.array(keys, np.uint64)
        packed[fn + ".offsets"] = np.cumsum([0] + [len(r) for r in rows]).astype(np.int64)
        packed[fn + ".data"] = np.concatenate(rows)
    np.savez_compressed(oracle.REF_ANSWERS, **packed)
    print("%d answers (%s) -> %s" % (len(answers), "reference" if REF else "restatement", oracle.REF_ANSWERS))


if __name__ == "__main__":
    main()
