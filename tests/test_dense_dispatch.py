"""Which kernel serves a matching call, at each coverage boundary of the sweeps (DESIGN §4, dispatch table).

Every job below sits just inside or just outside the coverage of a sweep. The test checks the kernel that
usv_last_kernel names and the kernel launches of one call. Launches are counted after a warm-up call of the same job,
because a context's first call also builds its distance table (one launch, once). A job that no kernel serves must be
refused with USV_ERR_UNSUPPORTED.

Launches of one call:
  - SAD sweep: 1; on colour frames 2 + 1 (the planes of both cameras, then the sweep);
  - correlation sweeps: 4 + 1 (row sums and window statistics of both cameras, then the sweep), plus 2 on colour frames;
  - direct form: 1;
  - the resolved disparity map: 1 more."""
import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, api

SAD = "dense_sad_argmin_kernel"
ALU = "dense_corr_argmin_kernel"
MMA = "dense_corr_mma_kernel"
UMMA = "dense_corr_umma_kernel"
DIRECT = "block_cost_argmin_direct"
REFUSED = None

# id: (frame w, h, channels, params, corr_kernel, extra outputs, sparse, kernel, launches)
CASES = {
    # gray SAD: template widths the SAD sweep covers (8 .. 32 in steps of 4, not 20) and those it does not
    "sad-tw4": (200, 64, 1, dict(tmpl_w=4), "auto", 0, False, DIRECT, 1),
    "sad-tw8": (200, 64, 1, dict(tmpl_w=8), "auto", 0, False, SAD, 1),
    "sad-tw12": (200, 64, 1, dict(tmpl_w=12), "auto", 0, False, SAD, 1),
    "sad-tw16": (200, 64, 1, dict(tmpl_w=16), "auto", 0, False, SAD, 1),
    "sad-tw20": (200, 64, 1, dict(tmpl_w=20), "auto", 0, False, DIRECT, 1),
    "sad-tw24": (200, 64, 1, dict(tmpl_w=24), "auto", 0, False, SAD, 1),
    "sad-tw32": (200, 64, 1, dict(tmpl_w=32), "auto", 0, False, SAD, 1),
    # template height: the SAD sweep and the ALU correlation sweep end at 64 rows
    "sad-th64": (200, 80, 1, dict(tmpl_h=64), "auto", 0, False, SAD, 1),
    "sad-th65": (200, 80, 1, dict(tmpl_h=65), "auto", 0, False, DIRECT, 1),
    # colour SAD: the SAD sweep, or the SAD arm of the ALU correlation kernel when that sweep is forced
    "sad-c3-auto": (200, 64, 3, dict(), "auto", 0, False, SAD, 3),
    "sad-c3-alu": (200, 64, 3, dict(), "alu", 0, False, ALU, 7),
    # forcing the ALU sweep leaves gray SAD on the SAD sweep, as does forcing a tensor-pipe sweep for any SAD
    "sad-gray-alu": (200, 64, 1, dict(), "alu", 0, False, SAD, 1),
    "sad-gray-mma": (200, 64, 1, dict(), "mma", 0, False, SAD, 1),
    "sad-c3-tcgen05": (200, 64, 3, dict(), "tcgen05", 0, False, SAD, 3),
    # the SAD key (cost << xb | candidate code) must fit 31 bits: beyond it, the SAD arm of the ALU correlation kernel
    "sad-key-32x64-w4094": (4094, 64, 1, dict(tmpl_w=32, tmpl_h=64), "auto", 0, False, SAD, 1),
    "sad-key-32x64-w4095": (4095, 64, 1, dict(tmpl_w=32, tmpl_h=64), "auto", 0, False, ALU, 5),
    "sad-key-c3-32x32-w2046": (2046, 32, 3, dict(tmpl_w=32, tmpl_h=32), "auto", 0, False, SAD, 3),
    "sad-key-c3-32x32-w2047": (2047, 32, 3, dict(tmpl_w=32, tmpl_h=32), "auto", 0, False, ALU, 7),
    # the dense sweeps take one or three channels, stride 1 and dense grids only
    "sad-c2": (200, 64, 2, dict(), "auto", 0, False, DIRECT, 1),
    "sad-c4": (200, 64, 4, dict(), "auto", 0, False, DIRECT, 1),
    "ncc-c2": (200, 64, 2, dict(cost="ncc"), "auto", 0, False, DIRECT, 1),
    "sad-stride-x2": (200, 64, 1, dict(stride_x=2), "auto", 0, False, DIRECT, 1),
    "ncc-stride-x2": (200, 64, 1, dict(cost="ncc", stride_x=2), "auto", 0, False, DIRECT, 1),
    "sad-sparse": (200, 64, 1, dict(), "auto", 0, True, DIRECT, 1),
    "ncc-sparse": (200, 64, 1, dict(cost="ncc"), "auto", 0, True, DIRECT, 1),
    # NCC: tcgen05 for gray frames of at least 128 windows a row, mma.sync below and on colour frames
    "ncc-nxc127": (142, 64, 1, dict(cost="ncc"), "auto", 0, False, MMA, 5),
    "ncc-nxc128": (143, 64, 1, dict(cost="ncc"), "auto", 0, False, UMMA, 5),
    "ncc-c3": (200, 64, 3, dict(cost="ncc"), "auto", 0, False, MMA, 7),
    "ssd-gray": (200, 64, 1, dict(cost="ssd"), "auto", 0, False, MMA, 5),
    # ZNCC template widths: the tensor-pipe sweeps take any width up to 32, the ALU sweep multiples of 4
    "zncc-tw5": (200, 64, 1, dict(cost="zncc", tmpl_w=5), "auto", 0, False, UMMA, 5),
    "zncc-tw32": (200, 64, 1, dict(cost="zncc", tmpl_w=32), "auto", 0, False, UMMA, 5),
    "zncc-tw36": (200, 64, 1, dict(cost="zncc", tmpl_w=36), "auto", 0, False, DIRECT, 1),
    # each forced sweep where it covers the job and where it does not
    "zncc-alu": (200, 64, 1, dict(cost="zncc"), "alu", 0, False, ALU, 5),
    "zncc-alu-tw5": (200, 64, 1, dict(cost="zncc", tmpl_w=5), "alu", 0, False, DIRECT, 1),
    "zncc-alu-th65": (200, 80, 1, dict(cost="zncc", tmpl_h=65), "alu", 0, False, DIRECT, 1),
    "zncc-mma": (200, 64, 1, dict(cost="zncc"), "mma", 0, False, MMA, 5),
    "zncc-mma-tw36": (200, 64, 1, dict(cost="zncc", tmpl_w=36), "mma", 0, False, DIRECT, 1),
    "ncc-c3-tcgen05": (200, 64, 3, dict(cost="ncc"), "tcgen05", 0, False, UMMA, 7),
    "ssd-tcgen05": (200, 64, 1, dict(cost="ssd"), "tcgen05", 0, False, UMMA, 5),
    "zncc-tcgen05-tw36": (200, 64, 1, dict(cost="zncc", tmpl_w=36), "tcgen05", 0, False, DIRECT, 1),
    # the resolved disparity map adds its own launch
    "sad-resolved": (200, 64, 1, dict(), "auto", _abi.OUT_RESOLVED_DISPARITY_U16, False, SAD, 2),
    "ncc-resolved": (200, 64, 1, dict(cost="ncc"), "auto", _abi.OUT_RESOLVED_DISPARITY_U16, False, UMMA, 6),
    # no kernel serves a one-pixel-wide template of 32 768 rows (the direct form cannot hold it in shared memory)
    "sad-tw1-th32768": (8, 32769, 1, dict(tmpl_w=1, tmpl_h=32768), "auto", 0, False, REFUSED, 0),
}


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _call(ctx, left, right, p, mask, sparse):
    if not sparse:
        return ctx.match_dense(left, right, p, mask=mask)
    tx = np.array([0, 5, 17, 100], np.int32)
    ty = np.array([0, 3, 40, 48], np.int32)
    return ctx.match_templates(left, right, tx, ty, p, mask=mask)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_kernel_and_launches_at_coverage_boundaries(ctx, case):
    w, h, c, kw, corr, extra, sparse, kernel, launches = CASES[case]
    rng = np.random.default_rng(len(case))
    shape = (1, h, w) if c == 1 else (1, h, w, c)
    left = rng.integers(0, 256, size=shape, dtype=np.uint8)
    right = np.roll(left, -3, axis=2)
    p = _abi.make_params(search_max=48, **kw)
    mask = api.ALL_OUTPUTS | extra
    ctx.corr_kernel(corr)
    try:
        if kernel is REFUSED:
            with pytest.raises(api.UsvError) as e:
                _call(ctx, left, right, p, mask, sparse)
            assert "(%d)" % _abi.USV_ERR_UNSUPPORTED in str(e.value), str(e.value)
            return
        _call(ctx, left, right, p, mask, sparse)  # warm-up: builds the distance table on the context's first call
        before = ctx.launch_count
        _call(ctx, left, right, p, mask, sparse)
        assert (ctx.last_kernel, ctx.launch_count - before) == (kernel, launches)
    finally:
        ctx.corr_kernel("auto")
