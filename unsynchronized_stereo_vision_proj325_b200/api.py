"""ctypes binding of libusv_b200.so (the C-ABI in include/usv_b200.h).

The library is the product; this module only marshals numpy / torch buffers
into it. There is no CPU fallback: if the shared library is missing or no
CUDA device is usable, the calls raise.
"""
import ctypes as C
import os
import weakref

import numpy as np

from . import _abi
from ._abi import FrameDesc, Outputs, SearchParams

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libusv_b200.so")

# every symbol include/usv_b200.h declares
EXPORTS = (
    "usv_abi_version", "usv_create", "usv_destroy", "usv_last_error", "usv_launch_count", "usv_last_kernel", "usv_device_status", "usv_set_option", "usv_distance_lut", "usv_block_search_host", "usv_stream_submit_io",
    "usv_grid_dims", "usv_match_dense_device", "usv_match_dense_host", "usv_match_templates_device",
    "usv_match_templates_host", "usv_disparity_to_distance", "usv_moving_object_distance",
    "usv_coordinate_position", "usv_pair_nearest", "usv_stream_create", "usv_stream_destroy",
    "usv_stream_slot", "usv_stream_frame_desc", "usv_stream_submit", "usv_stream_submit_from", "usv_stream_submit_gather",
    "usv_stream_wait", "usv_host_register", "usv_host_unregister",
    "usv_stream_bytes_per_pair", "usv_probe_issue_rate", "usv_match_contours",
    "usv_resolve_match_list", "usv_resolve_match_list_device", "usv_id_matcher", "usv_preprocess_device", "usv_preprocess_host",
    "usv_refine_subpixel_device", "usv_match_dense_subpixel_host",
)


class UsvError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libusv_b200.so; raise (never fall back) when it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise UsvError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.usv_last_error.restype = C.c_char_p
        L.usv_last_error.argtypes = [C.c_void_p]
        L.usv_last_kernel.restype = C.c_char_p
        L.usv_last_kernel.argtypes = [C.c_void_p]
        L.usv_launch_count.restype = C.c_int64
        L.usv_launch_count.argtypes = [C.c_void_p]
        L.usv_pair_nearest.restype = C.c_int64
        L.usv_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.usv_destroy.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(int(a))


def grid_dims(frame, params):
    """(nx, ny, candidate evaluations per pair) — pure host arithmetic."""
    nx, ny, ev = C.c_int32(), C.c_int32(), C.c_int64()
    rc = lib().usv_grid_dims(C.byref(frame), C.byref(params), C.byref(nx), C.byref(ny), C.byref(ev))
    if rc:
        raise UsvError("usv_grid_dims: invalid geometry (%d)" % rc)
    return nx.value, ny.value, ev.value


def pair_nearest(t_left, t_right, max_dt):
    """Host nearest-timestamp pairing (replaces the capture loop's timestamps,
    P/Main.cpp:876-905). Returns (left_idx, right_idx) int32 arrays."""
    tl = np.ascontiguousarray(t_left, np.float64)
    tr = np.ascontiguousarray(t_right, np.float64)
    cap = max(len(tl), 1)
    ol, orr = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
    n = lib().usv_pair_nearest(_ptr(tl), C.c_int64(len(tl)), _ptr(tr), C.c_int64(len(tr)), C.c_double(max_dt),
                               _ptr(ol), _ptr(orr), C.c_int64(cap))
    if n < 0:
        raise UsvError("usv_pair_nearest failed (%d): timestamps must be ascending" % n)
    return ol[:n].copy(), orr[:n].copy()


def _alloc_host_outputs(n, mask):
    arrs, st = {}, Outputs()
    for name, bit, dt in _abi.OUTPUT_FIELDS:
        if mask & bit:
            arrs[name] = np.zeros(n, dtype=dt)
            setattr(st, name, arrs[name].ctypes.data)
    return arrs, st


ALL_OUTPUTS = 0x7F


class Context:
    """One usv_ctx: a GPU plus its scratch buffers. Not thread-safe; create one
    per (GPU, host thread) as the header says."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = lib().usv_create(int(device), C.byref(self._h))
        if rc:
            self._h = None
            raise UsvError("usv_create(device=%d) failed with %d (%s)" % (
                device, rc, {-3: "no usable sm_100 CUDA device; there is no CPU fallback"}.get(rc, "see status codes")))
        self.device = device
        self._streams = weakref.WeakSet()  # open Streams: closed before the context (they borrow it)

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            for st in list(getattr(self, "_streams", ())):
                st.close()
            _lib.usv_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter teardown
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc:
            raise UsvError("%s failed (%d): %s" % (what, rc, lib().usv_last_error(self._h).decode()))

    def set_option(self, key, value):
        self._check(lib().usv_set_option(self._h, C.c_int32(int(key)), C.c_int64(int(value))), "usv_set_option")

    def corr_kernel(self, which):
        """Test / measurement aid: "auto" | "alu" | "mma" | "tcgen05" — the sweep that serves dense NCC / ZNCC / SSD."""
        self.set_option(1, {"auto": 0, "alu": 1, "mma": 2, "tcgen05": 3}[which])

    @property
    def launch_count(self):
        return lib().usv_launch_count(self._h)

    @property
    def last_kernel(self):
        return lib().usv_last_kernel(self._h).decode()

    # ---- host-buffer entry points -------------------------------------------
    def match_dense(self, left, right, params, mask=ALL_OUTPUTS):
        """left/right: [n, H, W(, C)] uint8 host arrays -> dict of [n, ny*nx]."""
        assert left.shape == right.shape and left.strides == right.strides
        f = _abi.frame_desc_for(left)
        nx, ny, _ = grid_dims(f, params)
        n = left.shape[0]
        arrs, st = _alloc_host_outputs(n * nx * ny, mask)
        rc = lib().usv_match_dense_host(self._h, _ptr(left), _ptr(right), C.byref(f), C.c_int32(n), C.byref(params), C.byref(st))
        self._check(rc, "usv_match_dense_host")
        return {k: v.reshape(n, ny * nx) for k, v in arrs.items()}

    def match_dense_subpixel(self, left, right, params, mask=ALL_OUTPUTS):
        """match_dense plus the sub-pixel refinement of its winners (usv_match_dense_subpixel_host): the same dict, plus
        "disparity_x16" (int32, 1/16 px, NO_SUBPIXEL where there is none) and "subpixel_distance" (f64, cm, from the
        refined disparity), each [n, ny*nx]."""
        assert left.shape == right.shape and left.strides == right.strides
        f = _abi.frame_desc_for(left)
        nx, ny, _ = grid_dims(f, params)
        n = left.shape[0]
        arrs, st = _alloc_host_outputs(n * nx * ny, mask)
        x16 = np.zeros(n * nx * ny, np.int32)
        dist = np.zeros(n * nx * ny, np.float64)
        rc = lib().usv_match_dense_subpixel_host(self._h, _ptr(left), _ptr(right), C.byref(f), C.c_int32(n), C.byref(params),
                                                 C.byref(st), _ptr(x16), _ptr(dist))
        self._check(rc, "usv_match_dense_subpixel_host")
        arrs["disparity_x16"], arrs["subpixel_distance"] = x16, dist
        return {k: v.reshape(n, ny * nx) for k, v in arrs.items()}

    def match_templates(self, left, right, tx, ty, params, mask=ALL_OUTPUTS, rows=False):
        assert left.shape == right.shape and left.strides == right.strides
        f = _abi.frame_desc_for(left)
        n, nt = left.shape[0], len(tx)
        tx = np.ascontiguousarray(tx, np.int32)
        ty = np.ascontiguousarray(ty, np.int32)
        arrs, st = _alloc_host_outputs(n * nt, mask)
        cap = f.width
        integer = params.cost_kind <= _abi.COST_SSD
        cost_rows = np.full((n, nt, cap), 0xFFFFFFFF, np.uint32) if rows and integer else None
        score_rows = np.full((n, nt, cap), np.nan, np.float64) if rows and not integer else None
        rc = lib().usv_match_templates_host(self._h, _ptr(left), _ptr(right), C.byref(f), C.c_int32(n), _ptr(tx), _ptr(ty),
                                            C.c_int32(nt), C.byref(params), C.byref(st), _ptr(cost_rows), _ptr(score_rows),
                                            C.c_int32(cap))
        self._check(rc, "usv_match_templates_host")
        out = {k: v.reshape(n, nt) for k, v in arrs.items()}
        if rows:
            out["cost_rows"], out["score_rows"] = cost_rows, score_rows
        return out

    def block_search(self, left, right, params):
        """One frame pair through the reference's call order on the device (usv_block_search_host): dense sweep -> the
        whole-list ResolveMatchList -> distance of every surviving record. left/right: [H, W(, C)] uint8.
        Returns (TentativeMatch as a MATCH_DTYPE array, distances f64)."""
        assert left.shape == right.shape and left.strides == right.strides
        f = _abi.frame_desc_for(left[None])
        nx, ny, _ = grid_dims(f, params)
        cap = nx * ny
        m = np.zeros(cap, _abi.MATCH_DTYPE)
        d = np.zeros(cap, np.float64)
        n = C.c_int64()
        rc = lib().usv_block_search_host(self._h, _ptr(left), _ptr(right), C.byref(f), C.byref(params), _ptr(m), _ptr(d), C.c_int64(cap), C.byref(n))
        self._check(rc, "usv_block_search_host")
        return m[:n.value], d[:n.value]

    # ---- device-pointer entry point (inputs resident in HBM) ------------------
    def match_dense_device(self, d_left, d_right, frame, n_pairs, params, d_out, stream=0):
        """Raw device pointers (ints); asynchronous on `stream` (a cudaStream_t)."""
        rc = lib().usv_match_dense_device(self._h, _ptr(d_left), _ptr(d_right), C.byref(frame), C.c_int32(n_pairs),
                                          C.byref(params), C.byref(d_out), C.c_void_p(int(stream)))
        self._check(rc, "usv_match_dense_device")

    def match_templates_device(self, d_left, d_right, frame, n_pairs, d_tx, d_ty, n_templates, params, d_out, stream=0,
                               d_cost_rows=None, d_score_rows=None, row_cap=0):
        """Raw device pointers (ints), explicit template list; asynchronous on `stream`."""
        rc = lib().usv_match_templates_device(self._h, _ptr(d_left), _ptr(d_right), C.byref(frame), C.c_int32(n_pairs), _ptr(d_tx),
                                              _ptr(d_ty), C.c_int32(n_templates), C.byref(params), C.byref(d_out), _ptr(d_cost_rows),
                                              _ptr(d_score_rows), C.c_int32(row_cap), C.c_void_p(int(stream)))
        self._check(rc, "usv_match_templates_device")

    def refine_subpixel_device(self, d_left, d_right, frame, n_pairs, params, d_right_index, d_disparity_x16, d_distance=None,
                               stream=0):
        """Sub-pixel refinement of dense winners, raw device pointers (ints); asynchronous on `stream`."""
        rc = lib().usv_refine_subpixel_device(self._h, _ptr(d_left), _ptr(d_right), C.byref(frame), C.c_int32(n_pairs),
                                              C.byref(params), _ptr(d_right_index), _ptr(d_disparity_x16), _ptr(d_distance),
                                              C.c_void_p(int(stream)))
        self._check(rc, "usv_refine_subpixel_device")

    # ---- distance family --------------------------------------------------------
    def disparity_to_distance(self, disp, kind):
        d = np.ascontiguousarray(disp, np.int32)
        out = np.zeros(d.shape, np.float64)
        self._check(lib().usv_disparity_to_distance(self._h, _ptr(d), C.c_int64(d.size), C.c_int32(kind), _ptr(out)),
                    "usv_disparity_to_distance")
        return out

    def distance_lut(self, kind, n):
        """distance[d] for d = 0 .. n-1, built on the device by the kernels' own epilogue function."""
        out = np.zeros(int(n), np.float64)
        self._check(lib().usv_distance_lut(self._h, C.c_int32(int(kind)), C.c_int32(int(n)), _ptr(out)), "usv_distance_lut")
        return out

    def moving_object_distance(self, camera_side, t_this, this_xy, other_xy, old_xy, older_xy, idx3, t_other, t_old, t_older):
        f32 = lambda a: np.ascontiguousarray(np.asarray(a, np.float32).reshape(-1, 2))  # noqa: E731
        this_xy, other_xy, old_xy, older_xy = map(f32, (this_xy, other_xy, old_xy, older_xy))
        idx3 = np.ascontiguousarray(np.asarray(idx3, np.int32).reshape(-1, 3))
        out = np.zeros(max(len(idx3), 1), np.float64)
        n_out = C.c_int32()
        rc = lib().usv_moving_object_distance(
            self._h, C.c_int32(int(camera_side)), C.c_int64(int(t_this)), _ptr(this_xy), C.c_int32(len(this_xy)),
            _ptr(other_xy), C.c_int32(len(other_xy)), _ptr(old_xy), C.c_int32(len(old_xy)), _ptr(older_xy),
            C.c_int32(len(older_xy)), _ptr(idx3), C.c_int32(len(idx3)), C.c_int64(int(t_other)), C.c_int64(int(t_old)),
            C.c_int64(int(t_older)), _ptr(out), C.byref(n_out))
        self._check(rc, "usv_moving_object_distance")
        return out[:n_out.value]

    def coordinate_position(self, camera_side, dist, xy):
        dist = np.ascontiguousarray(dist, np.float64)
        xy = np.ascontiguousarray(np.asarray(xy, np.float32).reshape(-1, 2))
        out = np.zeros((len(dist), 3), np.float64)
        self._check(lib().usv_coordinate_position(self._h, C.c_int32(int(camera_side)), _ptr(dist), _ptr(xy),
                                                  C.c_int64(len(dist)), _ptr(out)), "usv_coordinate_position")
        return out

    def match_contours(self, contours_this, contours_other, accept_threshold=0.75):
        """The reference's own GenerateMatchingList over contours (P/Main.cpp:403-426): lists of [n, 2] int
        arrays -> (matches in i-major / j-minor order, full cost matrix)."""
        def pack(cs):
            off = np.zeros(len(cs) + 1, np.int32)
            for i, c in enumerate(cs):
                off[i + 1] = off[i] + len(c)
            pts = np.zeros((max(int(off[-1]), 1), 2), np.int32)
            for i, c in enumerate(cs):
                pts[off[i]:off[i + 1]] = np.asarray(c, np.int32).reshape(-1, 2)
            return pts, off
        pl, ol = pack(contours_this)
        pr, orr = pack(contours_other)
        nl, nr = len(contours_this), len(contours_other)
        out = np.zeros(max(nl * nr, 1), _abi.MATCH_DTYPE)
        cm = np.zeros((max(nl, 1), max(nr, 1)), np.float64)
        n = C.c_int64()
        rc = lib().usv_match_contours(self._h, _ptr(pl), _ptr(ol), C.c_int32(nl), _ptr(pr), _ptr(orr), C.c_int32(nr),
                                      C.c_double(accept_threshold), _ptr(out), C.c_int64(len(out)), C.byref(n), _ptr(cm))
        self._check(rc, "usv_match_contours")
        return out[:n.value], cm[:nl, :nr]

    def resolve_match_list(self, matches, skip_unmatched=False):
        """ResolveMatchList (P/Main.cpp:432-477) on the GPU: MATCH_DTYPE array -> the reference's TentativeMatch."""
        m = np.ascontiguousarray(matches, dtype=_abi.MATCH_DTYPE)
        out = np.zeros(max(len(m), 1), dtype=_abi.MATCH_DTYPE)
        n = C.c_int64()
        rc = lib().usv_resolve_match_list(self._h, _ptr(m), C.c_int64(len(m)), C.c_int32(int(skip_unmatched)), _ptr(out),
                                          C.c_int64(len(out)), C.byref(n))
        self._check(rc, "usv_resolve_match_list")
        return out[:n.value]

    def id_matcher(self, cur, old):
        """IDMatcher (P/Main.cpp:483-499) on the GPU: two MATCH_DTYPE lists -> [n, 3] int32 triples."""
        a = np.ascontiguousarray(cur, dtype=_abi.MATCH_DTYPE)
        b = np.ascontiguousarray(old, dtype=_abi.MATCH_DTYPE)
        n = C.c_int64()
        rc = lib().usv_id_matcher(self._h, _ptr(a), C.c_int64(len(a)), _ptr(b), C.c_int64(len(b)), None, C.c_int64(0), C.byref(n))
        self._check(rc, "usv_id_matcher")
        out = np.zeros((max(n.value, 1), 3), np.int32)
        rc = lib().usv_id_matcher(self._h, _ptr(a), C.c_int64(len(a)), _ptr(b), C.c_int64(len(b)), _ptr(out), C.c_int64(len(out)), C.byref(n))
        self._check(rc, "usv_id_matcher")
        return out[:n.value]

    def preprocess(self, bgr, map1=None, map2=None, lighting=True, flavour=_abi.PRE_OPENCV4, dst_align=16):
        """The reference's pre-pass (P/Main.cpp:914-921) on the GPU: [n, H, W, 3] uint8 BGR frames (+ the fixed-point
        rectification maps) -> [n, H, W] uint8 gray frames (a view on rows padded to `dst_align` bytes)."""
        bgr = np.ascontiguousarray(bgr, np.uint8)
        assert bgr.ndim == 4 and bgr.shape[3] == 3
        n, h, w = bgr.shape[:3]
        pitch = -(-w // dst_align) * dst_align
        out = np.zeros((n, h, pitch), np.uint8)
        p = _abi.PreprocessParams(w, h, 3 * w, pitch, 3 * w * h, pitch * h, int(flavour), int(bool(lighting)))
        if map1 is not None:
            map1 = np.ascontiguousarray(map1, np.int16).reshape(h, w, 2)
            map2 = np.ascontiguousarray(map2, np.uint16).reshape(h, w)
        rc = lib().usv_preprocess_host(self._h, _ptr(bgr), C.c_int32(n), _ptr(map1), _ptr(map2), C.byref(p), _ptr(out))
        self._check(rc, "usv_preprocess_host")
        return out[:, :, :w]

    def preprocess_device(self, d_bgr, n_frames, d_map1, d_map2, params, d_gray, stream=0):
        rc = lib().usv_preprocess_device(self._h, _ptr(d_bgr), C.c_int32(n_frames), _ptr(d_map1), _ptr(d_map2), C.byref(params),
                                         _ptr(d_gray), C.c_void_p(int(stream)))
        self._check(rc, "usv_preprocess_device")

    def probe_issue_rate(self, which=0, target_ms=20.0):
        """Sustained thread-instructions/s of VABSDIFF4.U8.ACC (0) / IDP.4A (1): the ALU roofline denominator."""
        r = C.c_double()
        self._check(lib().usv_probe_issue_rate(self._h, C.c_int32(which), C.c_double(target_ms), C.byref(r)), "usv_probe_issue_rate")
        return r.value

    def host_register(self, array):
        """Page-lock a caller-owned numpy array (a frame store) so that copies from it are asynchronous."""
        self._check(lib().usv_host_register(self._h, _ptr(array), C.c_size_t(array.nbytes)), "usv_host_register")

    def host_unregister(self, array):
        self._check(lib().usv_host_unregister(self._h, _ptr(array)), "usv_host_unregister")

    def stream(self, frame, params, pairs_per_slot, n_slots=3, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_RAW_COST):
        return Stream(self, frame, params, pairs_per_slot, n_slots, mask)


class Stream:
    """Pinned ring of slots; each slot owns a CUDA stream: H2D -> kernels -> D2H
    overlap across slots (the replacement for the two capture threads)."""

    def __init__(self, ctx, frame, params, pairs_per_slot, n_slots, mask):
        self.ctx, self.params, self.mask = ctx, params, mask
        self.pairs_per_slot, self.n_slots = pairs_per_slot, n_slots
        self._h = C.c_void_p()
        rc = lib().usv_stream_create(ctx._h, C.byref(frame), C.byref(params), C.c_int32(pairs_per_slot), C.c_int32(n_slots),
                                     C.c_uint32(mask), C.byref(self._h))
        ctx._check(rc, "usv_stream_create")
        ctx._streams.add(self)
        self.frame = FrameDesc()
        lib().usv_stream_frame_desc(self._h, C.byref(self.frame))
        self.nx, self.ny, self.cand_evals = grid_dims(frame, params)
        h2d, d2h = C.c_int64(), C.c_int64()
        lib().usv_stream_bytes_per_pair(self._h, C.byref(h2d), C.byref(d2h))
        self.h2d_bytes_per_pair, self.d2h_bytes_per_pair = h2d.value, d2h.value
        self.slots = [self._slot_views(i) for i in range(n_slots)]

    def _slot_views(self, i):
        hl, hr, ho = C.c_void_p(), C.c_void_p(), Outputs()
        lib().usv_stream_slot(self._h, C.c_int32(i), C.byref(hl), C.byref(hr), C.byref(ho))
        f = self.frame
        nbytes = f.frame_stride * self.pairs_per_slot

        def view(p):
            buf = (C.c_uint8 * nbytes).from_address(p.value)
            a = np.frombuffer(buf, np.uint8).reshape(self.pairs_per_slot, f.height, f.row_stride)
            return a[:, :, : f.width * f.channels]

        outs = {}
        n_res = self.nx * self.ny * self.pairs_per_slot
        for name, bit, dt in _abi.OUTPUT_FIELDS:
            p = getattr(ho, name)
            if (self.mask & bit) and p:
                buf = (C.c_uint8 * (n_res * dt.itemsize)).from_address(p)
                outs[name] = np.frombuffer(buf, dt).reshape(self.pairs_per_slot, self.ny * self.nx)
        return {"left": view(hl), "right": view(hr), "out": outs}

    def submit(self, slot, n_pairs=None):
        n = self.pairs_per_slot if n_pairs is None else n_pairs
        self.ctx._check(lib().usv_stream_submit(self._h, C.c_int32(slot), C.c_int32(n)), "usv_stream_submit")

    def submit_from(self, slot, left, right, n_pairs=None):
        """Enqueue from caller-owned host arrays [n, H, W(, C)] (pinned for async copies)."""
        f = _abi.frame_desc_for(left)
        n = left.shape[0] if n_pairs is None else n_pairs
        self.ctx._check(lib().usv_stream_submit_from(self._h, C.c_int32(slot), _ptr(left), _ptr(right), C.byref(f), C.c_int32(n)),
                        "usv_stream_submit_from")

    def submit_gather(self, slot, left_store, idx_left, right_store, idx_right):
        """Enqueue pairs (left_store[idx_left[k]], right_store[idx_right[k]]) straight from two host frame stores
        [n, H, W(, C)] (register them with Context.host_register for asynchronous copies): no staging memcpy on the host."""
        f = _abi.frame_desc_for(left_store)
        il = np.ascontiguousarray(idx_left, np.int32)
        ir = np.ascontiguousarray(idx_right, np.int32)
        if len(il) != len(ir) or left_store.shape != right_store.shape:
            raise ValueError("index lists / frame stores differ in shape")
        self.ctx._check(lib().usv_stream_submit_gather(self._h, C.c_int32(slot), _ptr(left_store), _ptr(il), _ptr(right_store), _ptr(ir),
                                                       C.c_int64(left_store.shape[0]), C.byref(f), C.c_int32(len(il))),
                        "usv_stream_submit_gather")

    def submit_io(self, slot, left, right, outs):
        """Frames from, and results into, caller-owned host arrays (usv_stream_submit_io): `outs` maps output names of the
        stream's mask to C-contiguous arrays [n, ny*nx] that receive this submission's results directly."""
        f = _abi.frame_desc_for(left)
        st = Outputs()
        for name, bit, dt in _abi.OUTPUT_FIELDS:
            if self.mask & bit:
                a = outs[name]
                assert a.dtype == dt and a.flags["C_CONTIGUOUS"]
                setattr(st, name, a.ctypes.data)
        self.ctx._check(lib().usv_stream_submit_io(self._h, C.c_int32(slot), _ptr(left), _ptr(right), C.byref(f), C.c_int32(left.shape[0]), C.byref(st)),
                        "usv_stream_submit_io")

    def wait(self, slot):
        self.ctx._check(lib().usv_stream_wait(self._h, C.c_int32(slot)), "usv_stream_wait")

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            self.slots = []
            _lib.usv_stream_destroy(self._h)
            self.ctx._streams.discard(self)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter teardown
            pass
