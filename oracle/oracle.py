"""ctypes loader for the CPU oracle and the reference units compiled verbatim.

TEST INFRASTRUCTURE ONLY — imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs, never by the product package.
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

from unsynchronized_stereo_vision_proj325_b200 import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "_build", "libusv_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libusv_ref.so")
# the reference's answers on the inputs the tests give it (tests/golden/make_ref_answers.py): the ref_* functions
# below answer from this file when the reference's own code is not built, which is the case in any plain checkout
REF_ANSWERS = os.path.join(HERE, "..", "tests", "golden", "ref_answers.npz")


def build(quiet=True):
    """(Re)build oracle and, when /root/reference exists, oracle/_ref."""
    out = subprocess.run(["make", "-C", HERE, "all"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + out.stdout + out.stderr)
    if not quiet:
        print(out.stdout)


_lib = None
_ref = None
_P = C.POINTER


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def _same_cpu():
    """The oracle is compiled with -march=native; a copy built on a host with other ISA extensions must not be loaded."""
    sig = os.path.join(HERE, "_build", "cpu_flags.md5")
    try:
        import hashlib
        flags = next(l for l in open("/proc/cpuinfo") if l.startswith("flags"))
        return open(sig).read().split()[0] == hashlib.md5(flags.encode()).hexdigest()
    except Exception:
        return True


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, f) for f in ("block_search_oracle.c", "distance_oracle.c", "contour_oracle.c", "sliding_sad_cpu.c", "Makefile")]
        srcs.append(os.path.join(HERE, "..", "include", "usv_b200.h"))
        if _stale(ORACLE_SO, srcs) or not _same_cpu():
            if os.path.exists(ORACLE_SO):
                os.remove(ORACLE_SO)  # built with -march=native for another CPU (the .so travels to the GPU box): rebuild here
            build()
        L = C.CDLL(ORACLE_SO)
        L.usv_oracle_distance.restype = C.c_double
        L.usv_oracle_distance.argtypes = [C.c_int32, C.c_int32]
        L.usv_oracle_deg2rad.restype = C.c_double
        L.usv_oracle_deg2rad.argtypes = [C.c_double]
        L.usv_oracle_rad2deg.restype = C.c_double
        L.usv_oracle_rad2deg.argtypes = [C.c_double]
        L.usv_oracle_resolve_match_list.restype = C.c_int64
        L.usv_oracle_pair_nearest.restype = C.c_int64
        L.usv_oracle_id_matcher.restype = C.c_int64
        L.usv_oracle_match_contours.restype = C.c_int64
        L.usv_oracle_match_shapes_i1.restype = C.c_double
        L.usv_oracle_match_dense_sliding.restype = C.c_int64
        _lib = L
    return _lib


def ref():
    """The reference's own ResolveMatchList / DistanceCalculator.cpp, or None."""
    global _ref
    if _ref is None:
        if not os.path.exists(REF_SO):
            if os.path.isdir("/root/reference"):
                build()
            if not os.path.exists(REF_SO):
                return None
        R = C.CDLL(REF_SO)
        R.ref_resolve_match_list.restype = C.c_int64
        R.ref_id_matcher.restype = C.c_int64
        R.ref_deg2rad.restype = C.c_double
        R.ref_deg2rad.argtypes = [C.c_double]
        R.ref_rad2deg.restype = C.c_double
        R.ref_rad2deg.argtypes = [C.c_double]
        _ref = R
    return _ref


_answers = None


def answer_key(name, *inputs):
    """Key of one call of the reference in REF_ANSWERS: a 64-bit digest of the function's name and its inputs."""
    h = hashlib.sha256(name.encode())
    for a in inputs:
        a = np.ascontiguousarray(a)
        h.update(repr((a.shape, a.dtype.descr)).encode())
        h.update(a.tobytes())
    return int.from_bytes(h.digest()[:8], "little")


def recorded_answer(name, *inputs):
    """The reference's recorded answer to `name` on these inputs. REF_ANSWERS holds, per function, the keys of its
    calls, their answers concatenated along the first axis, and where each answer starts."""
    global _answers
    if _answers is None:
        _answers = {}
        with np.load(REF_ANSWERS) as z:
            for f in z.files:
                if f.endswith(".keys"):
                    fn = f[:-len(".keys")]
                    offsets, data = z[fn + ".offsets"], z[fn + ".data"]
                    for i, k in enumerate(z[f]):
                        _answers[fn, int(k)] = data[offsets[i]:offsets[i + 1]]
    key = answer_key(name, *inputs)
    if (name, key) not in _answers:
        raise LookupError("no recorded reference answer for this %s input (key %016x): build oracle/_ref from the reference "
                          "source, or record it with tests/golden/make_ref_answers.py" % (name, key))
    return _answers[name, key]


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def alloc_outputs(n, mask):
    """dict name -> numpy array for the requested output mask, plus the struct."""
    arrs, st = {}, _abi.Outputs()
    for name, bit, dt in _abi.OUTPUT_FIELDS:
        if mask & bit:
            arrs[name] = np.zeros(n, dtype=dt)
            setattr(st, name, arrs[name].ctypes.data)
    return arrs, st


ALL_OUTPUTS = 0x7F


def _with_cost_u16(arrs, mask, had_raw):
    """raw_cost_u16 (include/usv_b200.h): the u32 cost narrowed to 16 bits; ~0 (no candidate) becomes 0xFFFF."""
    if mask & _abi.OUT_RAW_COST_U16:
        rc = arrs["raw_cost"]
        assert (rc[rc != 0xFFFFFFFF] < 0xFFFF).all(), "raw_cost_u16 requested for costs that do not fit below 0xFFFF"
        arrs["raw_cost_u16"] = rc.astype(np.uint16)
        if not had_raw:
            del arrs["raw_cost"]
    return arrs


def grid_dims(frame, params):
    nx, ny, ev = C.c_int32(), C.c_int32(), C.c_int64()
    rc = lib().usv_oracle_grid_dims(C.byref(frame), C.byref(params), C.byref(nx), C.byref(ny), C.byref(ev))
    if rc:
        raise ValueError("bad geometry")
    return nx.value, ny.value, ev.value


def match_dense(left, right, params, mask=ALL_OUTPUTS, threads=0):
    """left/right: [n, H, W(, C)] uint8. Returns dict of arrays [n, ny*nx]."""
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    f = _abi.frame_desc_for(left)
    nx, ny, _ = grid_dims(f, params)
    n = left.shape[0]
    arrs, st = alloc_outputs(n * nx * ny, (mask & ~_abi.OUT_RAW_COST_U16) | (_abi.OUT_RAW_COST if mask & _abi.OUT_RAW_COST_U16 else 0))
    rc = lib().usv_oracle_match_dense(_ptr(left), _ptr(right), C.byref(f), C.c_int32(n), C.byref(params), C.byref(st), C.c_int32(threads))
    if rc:
        raise RuntimeError("oracle match_dense failed")
    arrs = _with_cost_u16(arrs, mask, bool(mask & _abi.OUT_RAW_COST))
    return {k: v.reshape(n, ny * nx) for k, v in arrs.items()}


def match_dense_rows(left, right, params, iy0, iy1, threads=0):
    """Bounded CPU-baseline sample: window rows [iy0, iy1) of one pair."""
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    f = _abi.frame_desc_for(left[None] if left.ndim in (2,) else left[None])
    nx, ny, _ = grid_dims(f, params)
    ri = np.zeros((iy1 - iy0) * nx, np.uint32)
    rc_ = np.zeros((iy1 - iy0) * nx, np.uint32)
    ev = C.c_int64()
    rc = lib().usv_oracle_match_dense_rows(_ptr(left), _ptr(right), C.byref(f), C.byref(params), C.c_int32(iy0), C.c_int32(iy1), _ptr(ri), _ptr(rc_), C.c_int32(threads), C.byref(ev))
    if rc:
        raise RuntimeError("oracle match_dense_rows failed")
    return ri, rc_, ev.value


def match_dense_sliding(left, right, params, iy0=0, iy1=None, threads=0):
    """The sliding-window CPU arm (sliding_sad_cpu.c): raw winners of window rows [iy0, iy1) of every pair.
    Returns (right_index [n, ny*nx], raw_cost [n, ny*nx], candidate evaluations done); rows outside stay NO_MATCH / ~0."""
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    f = _abi.frame_desc_for(left)
    nx, ny, _ = grid_dims(f, params)
    n = left.shape[0]
    iy1 = ny if iy1 is None else iy1
    ri = np.full(n * nx * ny, 0xFFFFFFFF, np.uint32)
    rc = np.full(n * nx * ny, 0xFFFFFFFF, np.uint32)
    ev = lib().usv_oracle_match_dense_sliding(_ptr(left), _ptr(right), C.byref(f), C.c_int32(n), C.byref(params), C.c_int32(iy0), C.c_int32(iy1),
                                              _ptr(ri), _ptr(rc), C.c_int32(threads))
    if ev < 0:
        raise RuntimeError("sliding CPU arm: unsupported job")
    return ri.reshape(n, ny * nx), rc.reshape(n, ny * nx), int(ev)


def match_templates(left, right, tx, ty, params, mask=ALL_OUTPUTS, rows=False):
    left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
    f = _abi.frame_desc_for(left)
    n, nt = left.shape[0], len(tx)
    tx = np.ascontiguousarray(tx, np.int32)
    ty = np.ascontiguousarray(ty, np.int32)
    arrs, st = alloc_outputs(n * nt, mask)
    cap = f.width
    cost_rows = np.full((n, nt, cap), 0xFFFFFFFF, np.uint32) if rows else None
    score_rows = np.full((n, nt, cap), np.nan, np.float64) if rows else None
    rc = lib().usv_oracle_match_templates(_ptr(left), _ptr(right), C.byref(f), C.c_int32(n), _ptr(tx), _ptr(ty), C.c_int32(nt), C.byref(params), C.byref(st), _ptr(cost_rows), _ptr(score_rows), C.c_int32(cap))
    if rc:
        raise RuntimeError("oracle match_templates failed")
    out = {k: v.reshape(n, nt) for k, v in arrs.items()}
    if rows:
        out["cost_rows"], out["score_rows"] = cost_rows, score_rows
    return out


def distance(disp, kind):
    return np.array([lib().usv_oracle_distance(int(d), int(kind)) for d in np.asarray(disp).ravel()], np.float64)


def _resolve(fn, matches):
    m = np.ascontiguousarray(matches, dtype=_abi.MATCH_DTYPE)
    out = np.zeros(max(len(m), 1), dtype=_abi.MATCH_DTYPE)
    n = fn(_ptr(m), C.c_int64(len(m)), _ptr(out), C.c_int64(len(out)))
    if n < 0:
        raise RuntimeError("resolve failed")
    return out[:n]


def resolve_match_list(matches):
    return _resolve(lib().usv_oracle_resolve_match_list, matches)


def ref_resolve_match_list(matches):
    if ref() is None:  # recorded as the input positions of the output records: every output record is an input record
        m = np.ascontiguousarray(matches, dtype=_abi.MATCH_DTYPE)
        return m[recorded_answer("resolve_match_list", m)]
    return _resolve(ref().ref_resolve_match_list, matches)


def _id_matcher(fn, cur, old):
    a = np.ascontiguousarray(cur, dtype=_abi.MATCH_DTYPE)
    b = np.ascontiguousarray(old, dtype=_abi.MATCH_DTYPE)
    cap = max(len(a) * len(b), 1)
    out = np.zeros((cap, 3), np.int32)
    n = fn(_ptr(a), C.c_int64(len(a)), _ptr(b), C.c_int64(len(b)), _ptr(out), C.c_int64(cap))
    if n < 0:
        raise RuntimeError("id matcher failed")
    return out[:n]


def id_matcher(cur, old):
    return _id_matcher(lib().usv_oracle_id_matcher, cur, old)


def ref_id_matcher(cur, old):
    if ref() is None:
        return recorded_answer("id_matcher", np.asarray(cur, _abi.MATCH_DTYPE), np.asarray(old, _abi.MATCH_DTYPE))
    return _id_matcher(ref().ref_id_matcher, cur, old)


def _f32(a):
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(-1, 2))


def _moving(fn, is_ref, camera_side, t_this, this_xy, other_xy, old_xy, older_xy, idx3, t_other, t_old, t_older):
    this_xy, other_xy, old_xy, older_xy = map(_f32, (this_xy, other_xy, old_xy, older_xy))
    idx3 = np.ascontiguousarray(np.asarray(idx3, np.int32).reshape(-1, 3))
    out = np.zeros(max(len(idx3), 1), np.float64)
    args = [C.c_int(int(camera_side)), C.c_int64(int(t_this)), _ptr(this_xy), C.c_int(len(this_xy)), _ptr(other_xy), C.c_int(len(other_xy)),
            _ptr(old_xy), C.c_int(len(old_xy)), _ptr(older_xy), C.c_int(len(older_xy)), _ptr(idx3), C.c_int(len(idx3)),
            C.c_int64(int(t_other)), C.c_int64(int(t_old)), C.c_int64(int(t_older)), _ptr(out)]
    if is_ref:
        args.append(C.c_int(len(out)))
    n = fn(*args)
    return out[:n]


def moving_object_distance(*a):
    return _moving(lib().usv_oracle_moving_object_distance, False, *a)


def ref_moving_object_distance(camera_side, t_this, this_xy, other_xy, old_xy, older_xy, idx3, t_other, t_old, t_older):
    if ref() is None:
        return recorded_answer("moving_object_distance", np.array([camera_side, t_this, t_other, t_old, t_older], np.int64),
                               *map(_f32, (this_xy, other_xy, old_xy, older_xy)), np.asarray(idx3, np.int32).reshape(-1, 3))
    return _moving(ref().ref_moving_object_distance, True, camera_side, t_this, this_xy, other_xy, old_xy, older_xy, idx3,
                   t_other, t_old, t_older)


def coordinate_position(camera_side, dist, xy):
    dist = np.ascontiguousarray(dist, np.float64)
    xy = _f32(xy)
    out = np.zeros((len(dist), 3), np.float64)
    lib().usv_oracle_coordinate_position(C.c_int(int(camera_side)), _ptr(dist), _ptr(xy), C.c_int64(len(dist)), _ptr(out))
    return out


def ref_coordinate_position(camera_side, dist, xy):
    dist = np.ascontiguousarray(dist, np.float64)
    xy = _f32(xy)
    if ref() is None:
        return recorded_answer("coordinate_position", np.int32(camera_side), dist, xy)
    out = np.zeros((len(dist), 3), np.float64)
    n = ref().ref_coordinate_position(C.c_int(int(camera_side)), _ptr(dist), _ptr(xy), C.c_int(len(dist)), _ptr(out))
    return out[:n]


def ref_sizeof_match():
    return int(recorded_answer("sizeof_match")[0]) if ref() is None else ref().ref_sizeof_match()


def ref_deg2rad(v):
    return float(recorded_answer("deg2rad", np.float64(v))[0]) if ref() is None else ref().ref_deg2rad(v)


def ref_rad2deg(v):
    return float(recorded_answer("rad2deg", np.float64(v))[0]) if ref() is None else ref().ref_rad2deg(v)


def pair_nearest(t_left, t_right, max_dt):
    tl = np.ascontiguousarray(t_left, np.float64)
    tr = np.ascontiguousarray(t_right, np.float64)
    ol = np.zeros(max(len(tl), 1), np.int32)
    orr = np.zeros(max(len(tl), 1), np.int32)
    n = lib().usv_oracle_pair_nearest(_ptr(tl), C.c_int64(len(tl)), _ptr(tr), C.c_int64(len(tr)), C.c_double(max_dt), _ptr(ol), _ptr(orr), C.c_int64(len(ol)))
    if n < 0:
        raise RuntimeError("pairing oracle failed")
    return ol[:n].copy(), orr[:n].copy()


CONTOUR_DESC = np.dtype([("hu", "<f8", (7,)), ("area", "<f8")])


def pack_contours(contours):
    """list of [n_i, 2] int arrays -> (concatenated int32 xy, int32 offsets)"""
    off = np.zeros(len(contours) + 1, np.int32)
    for i, c in enumerate(contours):
        off[i + 1] = off[i] + len(c)
    pts = np.zeros((max(int(off[-1]), 1), 2), np.int32)
    for i, c in enumerate(contours):
        pts[off[i]:off[i + 1]] = np.asarray(c, np.int32).reshape(-1, 2)
    return pts, off


def contour_descriptor(contour):
    c = np.ascontiguousarray(np.asarray(contour, np.int32).reshape(-1, 2))
    d = np.zeros(1, CONTOUR_DESC)
    lib().usv_oracle_contour_descriptor(_ptr(c), C.c_int32(len(c)), _ptr(d))
    return d[0]


def match_contours(contours_l, contours_r, threshold=0.75):
    """GenerateMatchingList over contours (P/Main.cpp:403-426). Returns (matches, cost matrix)."""
    pl, ol = pack_contours(contours_l)
    pr, orr = pack_contours(contours_r)
    nl, nr = len(contours_l), len(contours_r)
    out = np.zeros(max(nl * nr, 1), _abi.MATCH_DTYPE)
    cm = np.zeros((max(nl, 1), max(nr, 1)), np.float64)
    n = lib().usv_oracle_match_contours(_ptr(pl), _ptr(ol), C.c_int32(nl), _ptr(pr), _ptr(orr), C.c_int32(nr), C.c_double(threshold),
                                        _ptr(out), C.c_int64(len(out)), _ptr(cm))
    if n < 0:
        raise RuntimeError("contour oracle failed")
    return out[:n], cm[:nl, :nr]
